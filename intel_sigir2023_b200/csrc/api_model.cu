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
    INTEL_REQUIRE(d->bert_layers <= INTEL_MAX_BERT_LAYERS, INTEL_ERR_UNSUPPORTED, "too many BERT4Rec layers");
    return INTEL_OK;
}

// ================================================================================================
// self-attention stack (IntEL.py:182-197): N iterations sharing one set of weights
// ================================================================================================
struct StackWs {
    float* X[9];       // X[0] = input, X[l+1] = output of iteration l  (layers <= 8)
    float* QKV[8];
    float* A[8];
    float* U[8];
    float* Z[8];
    float* st[8];
};

void stack_layout(Arena& a, int64_t R, int d, int layers, StackWs& w) {
    w.X[0] = a.take<float>(R * d);
    for (int l = 0; l < layers; ++l) {
        w.QKV[l] = a.take<float>(R * 3 * d);
        w.A[l] = a.take<float>(R * d);
        w.U[l] = a.take<float>(R * d);
        w.Z[l] = a.take<float>(R * d);
        w.st[l] = a.take<float>(R * 2);
        w.X[l + 1] = a.take<float>(R * d);
    }
}

int g_use_fused_stack = 1;

int stack_fwd(int64_t B, int64_t L, int d, int heads, int layers, const intel_selfatt_t& p, StackWs& w, float drop_p,
              uint64_t drop_seed, int stream_id, cudaStream_t s, bool save = true) {
    const int64_t R = B * L;
    // whole stack of a session on chip: tcgen05 kernel (trunk_tc.cu, L <= 128) or the mma.sync kernel (trunk.cu, L <= 64);
    // both leave the same activations behind, which the fused and the staged backward passes read alike
    if (g_use_fused_stack && d == TD && trunk_fwd_supported(L, heads, layers)) {
        const StackParams sp{p.wq, p.wk, p.wv, p.w1, p.b1, p.w2, p.b2, p.lnw, p.lnb};
        const StackSaved sv{w.QKV, w.A, w.U, w.Z, w.st};
        return trunk_fwd(B, L, heads, layers, sp, w.X, sv, drop_p, drop_seed, stream_id, s, save);
    }
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
int stack_bwd(int64_t B, int64_t L, int d, int heads, int layers, const intel_selfatt_t& p, intel_selfatt_t& g,
              StackWs& w, float* dX, float* t1, float* t2, float* dqkv, float drop_p, uint64_t drop_seed, int stream_id,
              cudaStream_t s) {
    const int64_t R = B * L;
    if (g_use_fused_stack && trunk_supported(L, d, heads, layers)) {
        const StackParams sp{p.wq, p.wk, p.wv, p.w1, p.b1, p.w2, p.b2, p.lnw, p.lnb};
        const StackGrads sg{g.wq, g.wk, g.wv, g.w1, g.b1, g.w2, g.b2, g.lnw, g.lnb};
        const StackSaved sv{w.QKV, w.A, w.U, w.Z, w.st};
        return trunk_bwd(B, L, heads, layers, sp, sg, w.X, sv, dX, drop_p, drop_seed, stream_id, s);
    }
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
struct EnsWs {
    StackWs item, score;
    float* xs;                    // float copy of the scores [R,K]
    float *q_i, *q_s, *qk_i, *qk_s, *p_i, *p_s, *xbar_i, *xbar_s;   // cross attention
    // the three products that read the predicted intents ([B, I] x {query_layer (item), query_layer (score),
    // intent_embeddings}) run as one: Wcat [di + ds + dint, I] = the three weights stacked, qcat / dcat [B, di + ds + dint]
    float *Wcat, *qcat, *dcat;
    float* all;                   // [B, D] head input of the valid rows
    float *w_valid, *w_pad;       // [B,K]
    float *t_i, *t_s, *m_i, *m_s, *hu, *hint, *all_item;            // cross_attention = 0
    // backward scratch
    float *dall, *dwv, *dwp, *dxbar, *dqk, *dq, *dXa, *dXs, *t1, *t2, *dqkv;   // dXa / dXs: d(stack output) of the item / score stream
    float *g, *dall_item, *dm, *dt, *dvec;
};

void ens_layout(const intel_dims_t* d, Arena& a, EnsWs& w) {
    const int64_t B = d->B, L = d->L, R = B * L;
    const int di = d->d_iid + d->d_im, ds = d->d_s, D = di + ds + d->d_u + d->d_int;
    const int dmax = di > ds ? di : ds;
    stack_layout(a, R, di, d->layers, w.item);
    stack_layout(a, R, ds, d->layers, w.score);
    w.xs = a.take<float>(R * d->K);
    w.all = a.take<float>(B * D);
    w.w_valid = a.take<float>(B * d->K);
    w.w_pad = a.take<float>(B * d->K);
    w.dall = a.take<float>(B * D);
    w.dwv = a.take<float>(B * d->K);
    w.dwp = a.take<float>(B * d->K);
    w.dXa = a.take<float>(R * dmax);
    w.dXs = a.take<float>(R * dmax);
    w.t1 = a.take<float>(R * dmax);
    w.t2 = a.take<float>(R * dmax);
    w.dqkv = a.take<float>(R * 3 * dmax);
    if (d->cross_attention) {
        const int dc = di + ds + d->d_int;
        w.Wcat = a.take<float>((int64_t)dc * d->I);
        w.qcat = a.take<float>(B * dc);
        w.dcat = a.take<float>(B * dc);
        w.q_i = w.qcat; w.q_s = w.qcat + di;                    // column blocks of qcat (row stride dc)
        w.qk_i = a.take<float>(B * di); w.qk_s = a.take<float>(B * ds);
        w.p_i = a.take<float>(B * L); w.p_s = a.take<float>(B * L);
        w.xbar_i = a.take<float>(B * di); w.xbar_s = a.take<float>(B * ds);
        w.dxbar = a.take<float>(B * dmax);
        w.dqk = a.take<float>(B * dmax);
        w.dq = a.take<float>(B * dmax);
    } else {
        w.t_i = a.take<float>(B * d->qsize); w.t_s = a.take<float>(B * d->qsize);
        w.m_i = a.take<float>(B * di); w.m_s = a.take<float>(B * ds);
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
struct GruWs { float *gi, *h_all, *gates, *gh, *dh, *dgi, *dgh_all; int32_t *order, *rows_t, *rows_t1, *nlive; bool sorted; };   // sorted: set and read inside one call only
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
    EncWs e1, e2;
    float *feat, *logits, *dlogits, *dfeat;
    float *t1, *t2, *dqkv;   // bert backward scratch
};

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
        e.gru.gh = a.take<float>(B * 3 * h);
        e.gru.dh = a.take<float>(B * h);
        e.gru.dgi = a.take<float>(R * 3 * h);
        e.gru.dgh_all = a.take<float>(B * (T + 1) * 3 * h);
        e.gru.order = a.take<int32_t>(B + 1);
        e.gru.rows_t = a.take<int32_t>(R);
        e.gru.rows_t1 = a.take<int32_t>(R);
        e.gru.nlive = a.take<int32_t>(4);
    }
}

void int_layout(const intel_dims_t* d, Arena& a, IntWs& w) {
    const int d1 = d->d_ctx + d->d_int, d2 = d->d_iid + d->d_int;
    const int Dp = d1 + d2 + d->d_ctx + d->d_u;
    w.Wt = a.take<float>(d->I * d->d_int);
    w.dWt = a.take<float>(d->I * d->d_int);
    enc_layout(d, a, w.e1, d->H1, d1);
    enc_layout(d, a, w.e2, d->H2, d2);
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
int gru_fwd_pair(const intel_dims_t* d, const intel_encoder_t* const (&p)[2], EncWs* const (&e)[2], const int64_t* const (&lens)[2],
                 float* const (&out)[2], int64_t ld_out, cudaStream_t s) {
    const int64_t B = d->B;
    const int h = d->gru_hidden;
    bool fused = h == 128 && gru_tc_supported(h);
    {   // live rows and length order of both encoders: one launch
        int64_t Bs[2], Ts[2];
        const int64_t* ls[2];
        int32_t *rt[2], *rt1[2], *cn[2], *od[2];
        for (int i = 0; i < 2; ++i) {
            GruWs& w = e[i]->gru;
            Bs[i] = B; Ts[i] = e[i]->T; ls[i] = lens[i];
            const bool packed = B * (Ts[i] + 1) < (1LL << 31);
            rt[i] = packed ? w.rows_t : nullptr; rt1[i] = packed ? w.rows_t1 : nullptr; cn[i] = packed ? w.nlive : nullptr;
            w.sorted = Ts[i] <= 63;
            od[i] = w.sorted ? w.order : nullptr;
            fused = fused && w.sorted;
        }
        INTEL_TRY(gru_prep(2, Bs, Ts, ls, rt, rt1, cn, od, s));
    }
    for (int i = 0; i < 2; ++i) {
        const int64_t T = e[i]->T, R = B * T;
        const int dd = e[i]->d;
        GruWs& w = e[i]->gru;
        // the products over the [B, T] history rows walk the live rows only (about half of them are padding behind a
        // session's length; the reference packs the sequences: GeneralSeq.py:64-71).  gi rows of padding slots stay
        // unwritten: nobody reads them.
        const bool packed = B * (T + 1) < (1LL << 31);
        INTEL_TRY(linear(R, 3 * h, dd, e[i]->seq, dd, p[i]->w_ih, dd, p[i]->b_ih, w.gi, 3 * h, s, false, false, nullptr, 0,
                         packed ? w.rows_t : nullptr, packed ? w.nlive : nullptr));
        if (h == 128) {
            // the fused kernels write h_all[:, 1..T] of every session themselves: only the initial state h_0 needs clearing
            // (2 MB instead of a 44 MB memset per encoder and step)
            cudaError_t ce = cudaMemset2DAsync(w.h_all, (size_t)(T + 1) * h * 4, 0, (size_t)h * 4, (size_t)B, s);
            INTEL_REQUIRE(ce == cudaSuccess, INTEL_ERR_CUDA, "cudaMemset2DAsync: %s", cudaGetErrorString(ce));
        } else {
            INTEL_TRY(fill_zero(w.h_all, (size_t)B * (T + 1) * h * 4, s));
        }
    }
    if (fused) {
        GruTcPair pr;
        pr.n = 2;
        for (int i = 0; i < 2; ++i) {
            GruWs& w = e[i]->gru;
            pr.e[i] = GruTcOne{B, e[i]->T, lens[i], w.gi, p[i]->w_hh, p[i]->b_hh, w.h_all, w.gates, w.order};
        }
        INTEL_TRY(gru_tc_fwd_pair(pr, s, d->inference == 0));
    } else {
        for (int i = 0; i < 2; ++i) {
            const int64_t T = e[i]->T;
            GruWs& w = e[i]->gru;
            if (h == 128) {
                INTEL_TRY(gru_seq_fwd(B, T, h, lens[i], w.gi, p[i]->w_hh, p[i]->b_hh, w.h_all, w.gates, s, d->inference == 0));
            } else {
                for (int64_t t = 0; t < T; ++t) {
                    INTEL_TRY(linear(B, 3 * h, h, w.h_all + t * h, (T + 1) * h, p[i]->w_hh, h, p[i]->b_hh, w.gh, 3 * h, s));
                    INTEL_TRY(gru_step_fwd(B, T, h, (int)t, lens[i], w.gi, w.gh, w.h_all, w.gates, s));
                }
            }
        }
    }
    if (gru_outproj_pair_ok(h, e[0]->d, e[1]->d)) {          // both output projections in one launch
        const int n[2] = {e[0]->d, e[1]->d};
        const float* W[2] = {p[0]->w_out, p[1]->w_out};
        const float* hl[2] = {e[0]->gru.h_all + e[0]->T * h, e[1]->gru.h_all + e[1]->T * h};
        const int64_t ldh[2] = {(e[0]->T + 1) * h, (e[1]->T + 1) * h}, ldo[2] = {ld_out, ld_out};
        return gru_outproj_pair_fwd(B, n, W, hl, ldh, out, ldo, s);
    }
    for (int i = 0; i < 2; ++i) {
        const int64_t T = e[i]->T;
        GruWs& w = e[i]->gru;
        INTEL_TRY(linear(B, e[i]->d, h, w.h_all + T * h, (T + 1) * h, p[i]->w_out, h, nullptr, out[i], ld_out, s));
    }
    return INTEL_OK;
}

// have_dh: d(last state) was already formed (for both encoders at once, gru_outproj_pair_dx)
int gru_bwd(const intel_dims_t* d, const intel_encoder_t& p, intel_encoder_t& g, EncWs& e, const int64_t* lens,
            const float* dout, int64_t ld, cudaStream_t s, bool have_dh = false) {
    const int64_t B = d->B, T = e.T, R = B * T;
    const int dd = e.d, h = d->gru_hidden;
    GruWs& w = e.gru;
    INTEL_TRY(linear_dw(B, dd, h, dout, ld, w.h_all + T * h, (T + 1) * h, g.w_out, h, nullptr, s));
    if (!have_dh) INTEL_TRY(linear_dx(B, dd, h, dout, ld, p.w_out, h, w.dh, h, s));
    if (h == 128) {
        // the fused kernel writes dgh_all[:, 0..T-1] of every session (zeros behind a session's end): only slot T, which
        // pairs with the final state in the weight-gradient product below, needs clearing (6 MB instead of 132 MB)
        cudaError_t ce = cudaMemset2DAsync(w.dgh_all + T * 3 * h, (size_t)(T + 1) * 3 * h * 4, 0, (size_t)3 * h * 4, (size_t)B, s);
        INTEL_REQUIRE(ce == cudaSuccess, INTEL_ERR_CUDA, "cudaMemset2DAsync: %s", cudaGetErrorString(ce));
        // the fused kernel also sums the bias gradients (column sums of dgi / dgh) on its way
        int32_t* order = nullptr;
        if (T <= 63) {               // tiles of equally long sessions: a tile stops at its own last step
            INTEL_TRY(fill_zero(w.order + B, sizeof(int32_t), s));     // the order is the forward call's; reset the tile counter
            order = w.order;
        }
        INTEL_TRY(gru_seq_bwd(B, T, h, lens, p.w_hh, w.h_all, w.gates, w.dh, w.dgi, w.dgh_all, g.b_ih, g.b_hh, s, order));
    } else {
        INTEL_TRY(fill_zero(w.dgh_all, (size_t)B * (T + 1) * 3 * h * 4, s));
        for (int64_t t = T - 1; t >= 0; --t) {
            INTEL_TRY(gru_step_bwd(B, T, h, (int)t, lens, w.h_all, w.gates, w.dh, w.dgi, w.dgh_all, s));
            INTEL_TRY(linear_dx(B, 3 * h, h, w.dgh_all + t * 3 * h, (T + 1) * 3 * h, p.w_hh, h, w.dh, h, s, 1));
        }
    }
    // gradient rows of padding slots are zero: the three products below contract / map the live rows only (the list was
    // built by the forward call); d(seq) of the padding slots is cleared for the scatters that read every row
    const bool packed = B * (T + 1) < (1LL << 31);
    const int32_t *rt = packed ? w.rows_t : nullptr, *rt1 = packed ? w.rows_t1 : nullptr, *nl = packed ? w.nlive : nullptr;
    INTEL_TRY(linear_dw(B * (T + 1), 3 * h, h, w.dgh_all, 3 * h, w.h_all, h, g.w_hh, h, h == 128 ? nullptr : g.b_hh, s, false, rt1, nl));
    INTEL_TRY(linear_dw(R, 3 * h, dd, w.dgi, 3 * h, e.seq, dd, g.w_ih, dd, h == 128 ? nullptr : g.b_ih, s, false, rt, nl));
    if (packed) INTEL_TRY(fill_zero(e.dseq, (size_t)R * dd * 4, s));
    return linear_dx(R, 3 * h, dd, w.dgi, 3 * h, p.w_ih, dd, e.dseq, dd, s, 0, nullptr, 0, rt, nl);
}

}  // namespace

extern "C" {

int intel_debug_use_fused_stack(int on) {
    g_use_fused_stack = on ? 1 : 0;
    return INTEL_OK;
}

int intel_debug_use_tcgen05_gemm(int on) {
    gemm_debug_use_umma(on);
    return INTEL_OK;
}

int intel_debug_use_rows_gemm(int on) {
    gemm_debug_use_rows_tc(on);
    gemm_debug_use_wgrad_tc(on);
    return INTEL_OK;
}

int intel_debug_gru_prep(int64_t B, int64_t T, const int64_t* lens, int32_t* order, int32_t* rows_t, int32_t* rows_t1,
                         int32_t* count, intel_stream_t stream) {
    INTEL_REQUIRE(lens && order && rows_t && rows_t1 && count, INTEL_ERR_ARG, "gru_prep: null argument");
    return gru_prep(1, &B, &T, &lens, &rows_t, &rows_t1, &count, &order, S(stream));
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

    // embedding gathers straight into the concatenated item-stream rows (IntEL.py:170-175)
    INTEL_TRY(gather_rows(R, d->d_iid, P->iid_emb, bt->i_id, w.item.X[0], di, 0, s, d->item_rows));
    if (d->d_im > 0) INTEL_TRY(gather_rows(R, d->d_im, P->item_emb, bt->i_class, w.item.X[0] + d->d_iid, di, 0, s, d->class_rows));
    INTEL_TRY(score_embed_fwd(R, K, ds, bt->scores, P->score_w, P->score_b, w.score.X[0], w.xs, s));
    INTEL_TRY(stack_fwd(B, L, di, d->heads, d->layers, P->item, w.item, d->dropout_p, d->dropout_seed, 0, s, d->inference == 0));
    INTEL_TRY(stack_fwd(B, L, ds, d->heads, d->layers, P->score, w.score, d->dropout_p, d->dropout_seed, 1, s, d->inference == 0));
    float* Xi = w.item.X[d->layers];
    float* Xs = w.score.X[d->layers];

    if (d->cross_attention) {
        const float scale = 1.0f / sqrtf((float)d->qsize);
        // q_item | q_score | intent_embeddings(intent): one product over the predicted intents (read once instead of
        // three times); the weights are stacked into Wcat unless the caller already keeps them back to back
        const int dc = di + ds + dint;
        const float* Wc = P->xq_item;
        if (!(P->xq_score == P->xq_item + (int64_t)di * I && P->intent_w == P->xq_score + (int64_t)ds * I)) {
            INTEL_TRY(copy_d2d(w.Wcat, P->xq_item, (size_t)di * I * 4, s));
            INTEL_TRY(copy_d2d(w.Wcat + (int64_t)di * I, P->xq_score, (size_t)ds * I * 4, s));
            INTEL_TRY(copy_d2d(w.Wcat + (int64_t)(di + ds) * I, P->intent_w, (size_t)dint * I * 4, s));
            Wc = w.Wcat;
        }
        INTEL_TRY(linear(B, dc, I, intents, I, Wc, I, nullptr, w.qcat, dc, s));
        // item stream, score stream: qk = W_k^T q, the pooling, the value projection into the head input
        if (cross_full_ok(di, L) && al16(P->xk_item) && al16(P->xv_item)) {
            INTEL_TRY(cross_full_fwd(B, L, Xi, w.q_i, dc, P->xk_item, P->xv_item, bt->session_len, scale, w.p_i, w.qk_i, w.xbar_i, w.all, D, s));
        } else {
            INTEL_TRY(linear_dx(B, di, di, w.q_i, dc, P->xk_item, di, w.qk_i, di, s));            // qk = W_k^T q
            INTEL_TRY(cross_pool_fwd(B, L, di, Xi, w.qk_i, bt->session_len, scale, w.p_i, w.xbar_i, s));
            INTEL_TRY(linear(B, di, di, w.xbar_i, di, P->xv_item, di, nullptr, w.all, D, s));
        }
        if (cross_full_ok(ds, L) && al16(P->xk_score) && al16(P->xv_score)) {
            INTEL_TRY(cross_full_fwd(B, L, Xs, w.q_s, dc, P->xk_score, P->xv_score, bt->session_len, scale, w.p_s, w.qk_s, w.xbar_s,
                                     w.all + di, D, s));
        } else {
            INTEL_TRY(linear_dx(B, ds, ds, w.q_s, dc, P->xk_score, ds, w.qk_s, ds, s));
            INTEL_TRY(cross_pool_fwd(B, L, ds, Xs, w.qk_s, bt->session_len, scale, w.p_s, w.xbar_s, s));
            INTEL_TRY(linear(B, ds, ds, w.xbar_s, ds, P->xv_score, ds, nullptr, w.all + di, D, s));
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
        INTEL_TRY(linear(B, q, I, intents, I, P->gate_item_w0, I, P->gate_item_b0, w.t_i, q, s, false, true));
        INTEL_TRY(linear(B, di, q, w.t_i, q, P->gate_item_w2, q, nullptr, w.m_i, di, s));
        INTEL_TRY(linear(B, q, I, intents, I, P->gate_score_w0, I, P->gate_score_b0, w.t_s, q, s, false, true));
        INTEL_TRY(linear(B, ds, q, w.t_s, q, P->gate_score_w2, q, nullptr, w.m_s, ds, s));
        INTEL_TRY(gate_fwd(B, L, di, Xi, w.m_i, w.all_item, D, s));
        INTEL_TRY(gate_fwd(B, L, ds, Xs, w.m_s, w.all_item + di, D, s));
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
    float* Xi = w.item.X[d->layers];
    float* Xs = w.score.X[d->layers];

    float* const dXst[2] = {w.dXa, w.dXs};
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
            const int dd = st == 0 ? di : ds;
            const int off = st == 0 ? 0 : di;
            float* X = st == 0 ? Xi : Xs;
            float *q = st == 0 ? w.q_i : w.q_s, *qk = st == 0 ? w.qk_i : w.qk_s, *p = st == 0 ? w.p_i : w.p_s;
            float* xbar = st == 0 ? w.xbar_i : w.xbar_s;
            const float *xq = st == 0 ? P->xq_item : P->xq_score, *xk = st == 0 ? P->xk_item : P->xk_score,
                        *xv = st == 0 ? P->xv_item : P->xv_score;
            float *gxq = st == 0 ? G->xq_item : G->xq_score, *gxk = st == 0 ? G->xk_item : G->xk_score,
                  *gxv = st == 0 ? G->xv_item : G->xv_score;
            if (cross_full_ok(dd, L) && al16(xk) && al16(xv)) {
                INTEL_TRY(cross_full_bwd(B, L, X, q, dc, qk, xk, xv, bt->session_len, scale, p, xbar, w.dall + off, D, dXst[st],
                                         w.dcat + off, dc, gxk, gxv, s));
            } else {
                INTEL_TRY(linear_dw(B, dd, dd, w.dall + off, D, xbar, dd, gxv, dd, nullptr, s));
                INTEL_TRY(linear_dx(B, dd, dd, w.dall + off, D, xv, dd, w.dxbar, dd, s));
                INTEL_TRY(cross_pool_bwd(B, L, dd, X, qk, bt->session_len, scale, p, w.dxbar, dXst[st], w.dqk, s));
                INTEL_TRY(linear_dw(B, dd, dd, q, dc, w.dqk, dd, gxk, dd, nullptr, s));            // dW_k[a,c] = sum q_a dqk_c
                INTEL_TRY(linear(B, dd, dd, w.dqk, dd, xk, dd, nullptr, w.dcat + off, dc, s));      // dq = W_k dqk -> its block of dcat
            }
            (void)xq; (void)gxq;
        }
        // the three products against the predicted intents as one: d_intents = dcat Wcat, dWcat += dcat^T intents
        {
            const float* Wc = P->xq_item;
            if (!(P->xq_score == P->xq_item + (int64_t)di * I && P->intent_w == P->xq_score + (int64_t)ds * I)) Wc = w.Wcat;   // stacked by the forward call
            INTEL_TRY(linear_dx(B, dc, I, w.dcat, dc, Wc, I, d_intents_out, I, s, 0));
            if (G->xq_score == G->xq_item + (int64_t)di * I && G->intent_w == G->xq_score + (int64_t)ds * I) {
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
            const int dd = st == 0 ? di : ds;
            const int off = st == 0 ? 0 : di;
            float* X = st == 0 ? Xi : Xs;
            float *m = st == 0 ? w.m_i : w.m_s, *t = st == 0 ? w.t_i : w.t_s;
            const float *w0 = st == 0 ? P->gate_item_w0 : P->gate_score_w0, *w2 = st == 0 ? P->gate_item_w2 : P->gate_score_w2;
            float *gw0 = st == 0 ? G->gate_item_w0 : G->gate_score_w0, *gb0 = st == 0 ? G->gate_item_b0 : G->gate_score_b0,
                  *gw2 = st == 0 ? G->gate_item_w2 : G->gate_score_w2;
            INTEL_TRY(gate_bwd(B, L, dd, X, m, w.dall_item + off, D, dXst[st], w.dm, s));
            INTEL_TRY(linear_dw(B, dd, q, w.dm, dd, t, q, gw2, q, nullptr, s));
            INTEL_TRY(linear_dx(B, dd, q, w.dm, dd, w2, q, w.dt, q, s, 0, t, q));       // relu mask (t = relu(.) > 0)
            INTEL_TRY(linear_dw(B, q, I, w.dt, q, intents, I, gw0, I, gb0, s));
            INTEL_TRY(linear_dx(B, q, I, w.dt, q, w0, I, d_intents_out, I, s, 1));
        }
        }
    }
    // the self-attention stacks (IntEL.py:182-197) and what feeds them
    if (do_item) {
        INTEL_TRY(stack_bwd(B, L, di, d->heads, d->layers, P->item, G->item, w.item, w.dXa, w.t1, w.t2, w.dqkv, d->dropout_p,
                            d->dropout_seed, 0, s));
        INTEL_TRY(scatter_add_rows(R, d->d_iid, w.dXa, di, bt->i_id, G->iid_emb, nullptr, s, d->item_rows, M.iid));
        if (d->d_im > 0)
            INTEL_TRY(scatter_add_rows(R, d->d_im, w.dXa + d->d_iid, di, bt->i_class, G->item_emb, nullptr, s, d->class_rows, M.item));
    }
    if (do_score) {
        // run on its own, this phase is the one a caller overlaps with its gradient exchange: leave the reserved SMs free
        trunk_reserve_apply(phases == INTEL_ENS_BWD_SCORE);
        const int st = stack_bwd(B, L, ds, d->heads, d->layers, P->score, G->score, w.score, w.dXs, w.t1, w.t2, w.dqkv, d->dropout_p,
                                 d->dropout_seed, 1, s);
        trunk_reserve_apply(false);
        INTEL_TRY(st);
        if (score_embed_bwd_ok(K, ds)) INTEL_TRY(score_embed_bwd(R, K, ds, w.dXs, ds, w.xs, G->score_w, G->score_b, s));
        else INTEL_TRY(linear_dw(R, ds, K, w.dXs, ds, w.xs, K, G->score_w, K, G->score_b, s));
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
    const int dint = d->d_int, dctx = d->d_ctx, du = d->d_u, diid = d->d_iid;
    const int d1 = dctx + dint, d2 = diid + dint, Dp = d1 + d2 + dctx + du;
    const int off_v2 = dctx + du, off_v1 = dctx + du + d2;     // pred_layer input = [ctx | user | item-history | history]

    INTEL_TRY(transpose(dint, I, P->intent_w, w.Wt, 0, s));
    // session history tokens: [context embedding | intent embedding of the dense history intents]
    INTEL_TRY(gather_rows(B * d->H1, dctx, P->ctx_emb, bt->his_context, w.e1.seq, d1, 0, s, d->ctx_rows));
    if (bt->his_intents_idx) {
        INTEL_TRY(sparse_rows_linear_fwd(B * d->H1, bt->nz1, dint, bt->his_intents_idx, bt->his_intents_val, w.Wt,
                                         P->intent_b, w.e1.seq + dctx, d1, s));
    } else {
        INTEL_REQUIRE(bt->his_intents, INTEL_ERR_ARG, "his_intents is null");
        INTEL_TRY(dense_rows_linear_fwd(B * d->H1, I, dint, bt->his_intents, w.Wt, P->intent_b, w.e1.seq + dctx, d1,
                                        w.e1.nz_idx, w.e1.nz_val, w.e1.nz_cnt, NZ_CAP, s, d->H1, bt->history_len));
    }
    // item history tokens: [item id embedding | intent embedding of the one-hot item intents]
    INTEL_TRY(gather_rows(B * d->H2, diid, P->iid_emb, bt->his_item_id, w.e2.seq, d2, 0, s, d->item_rows));
    if (bt->his_item_int_idx) {
        INTEL_TRY(sparse_rows_linear_fwd(B * d->H2, bt->nz2, dint, bt->his_item_int_idx, bt->his_item_int_val, w.Wt,
                                         P->intent_b, w.e2.seq + diid, d2, s));
    } else {
        INTEL_REQUIRE(bt->his_item_int, INTEL_ERR_ARG, "his_item_int is null");
        INTEL_TRY(dense_rows_linear_fwd(B * d->H2, I, dint, bt->his_item_int, w.Wt, P->intent_b, w.e2.seq + diid, d2,
                                        w.e2.nz_idx, w.e2.nz_val, w.e2.nz_cnt, NZ_CAP, s, d->H2, bt->history_item_len));
    }
    if (d->encoder == INTEL_ENCODER_BERT4REC) {
        INTEL_TRY(bert_fwd(d, P->enc, w.e1, bt->history_len, w.feat + off_v1, Dp, s));
        INTEL_TRY(bert_fwd(d, P->item_enc, w.e2, bt->history_item_len, w.feat + off_v2, Dp, s));
    } else {
        const intel_encoder_t* const pe[2] = {&P->enc, &P->item_enc};
        EncWs* const ee[2] = {&w.e1, &w.e2};
        const int64_t* const ll[2] = {bt->history_len, bt->history_item_len};
        float* const oo[2] = {w.feat + off_v1, w.feat + off_v2};
        INTEL_TRY(gru_fwd_pair(d, pe, ee, ll, oo, Dp, s));
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
    const int dint = d->d_int, dctx = d->d_ctx, du = d->d_u, diid = d->d_iid;
    const int d1 = dctx + dint, d2 = diid + dint, Dp = d1 + d2 + dctx + du;
    const int off_v2 = dctx + du, off_v1 = dctx + du + d2;

    INTEL_TRY(softmax_rows_bwd(B, I, intents, d_intents, d_intents_extra, w.dlogits, s, pad4(I)));
    INTEL_TRY(linear_dw(B, I, Dp, w.dlogits, pad4(I), w.feat, Dp, G->pred_w, Dp, G->pred_b, s));
    INTEL_TRY(linear_dx(B, I, Dp, w.dlogits, pad4(I), P->pred_w, Dp, w.dfeat, Dp, s));
    INTEL_TRY(scatter_add_rows(B, dctx, w.dfeat, Dp, bt->context_mh, G->ctx_emb, nullptr, s, d->ctx_rows, M.ctx));
    INTEL_TRY(scatter_add_rows(B, du, w.dfeat + dctx, Dp, bt->u_id, G->uid_emb, nullptr, s, d->user_rows, M.uid));
    if (d->encoder == INTEL_ENCODER_BERT4REC) {
        INTEL_TRY(bert_bwd(d, P->enc, G->enc, w.e1, bt->history_len, w.dfeat + off_v1, Dp, w.t1, w.t2, w.dqkv, s));
        INTEL_TRY(bert_bwd(d, P->item_enc, G->item_enc, w.e2, bt->history_item_len, w.dfeat + off_v2, Dp, w.t1, w.t2, w.dqkv, s));
    } else {
        bool have_dh = false;
        if (gru_outproj_pair_ok(d->gru_hidden, w.e1.d, w.e2.d)) {      // d(last state) of both encoders in one launch
            const int n[2] = {w.e1.d, w.e2.d};
            const float* W[2] = {P->enc.w_out, P->item_enc.w_out};
            const float* dv[2] = {w.dfeat + off_v1, w.dfeat + off_v2};
            float* dh[2] = {w.e1.gru.dh, w.e2.gru.dh};
            const int64_t ldd[2] = {Dp, Dp}, ldh[2] = {d->gru_hidden, d->gru_hidden};
            INTEL_TRY(gru_outproj_pair_dx(B, n, W, dv, ldd, dh, ldh, s));
            have_dh = true;
        }
        INTEL_TRY(gru_bwd(d, P->enc, G->enc, w.e1, bt->history_len, w.dfeat + off_v1, Dp, s, have_dh));
        INTEL_TRY(gru_bwd(d, P->item_enc, G->item_enc, w.e2, bt->history_item_len, w.dfeat + off_v2, Dp, s, have_dh));
    }
    INTEL_TRY(fill_zero(w.dWt, (size_t)I * dint * 4, s));
    INTEL_TRY(scatter_add_rows(B * d->H1, dctx, w.e1.dseq, d1, bt->his_context, G->ctx_emb, nullptr, s, d->ctx_rows, M.ctx));
    if (bt->his_intents_idx) {
        INTEL_TRY(dense_rows_linear_bwd(B * d->H1, I, dint, nullptr, w.e1.dseq + dctx, d1, bt->his_intents_idx,
                                        bt->his_intents_val, nullptr, bt->nz1, w.dWt, s, G->intent_b));
    } else {
        INTEL_TRY(dense_rows_linear_bwd(B * d->H1, I, dint, bt->his_intents, w.e1.dseq + dctx, d1, w.e1.nz_idx, w.e1.nz_val,
                                        w.e1.nz_cnt, NZ_CAP, w.dWt, s, G->intent_b));      // + the bias gradient (column sums)
    }
    INTEL_TRY(scatter_add_rows(B * d->H2, diid, w.e2.dseq, d2, bt->his_item_id, G->iid_emb, nullptr, s, d->item_rows, M.iid));
    if (bt->his_item_int_idx) {
        INTEL_TRY(dense_rows_linear_bwd(B * d->H2, I, dint, nullptr, w.e2.dseq + diid, d2, bt->his_item_int_idx,
                                        bt->his_item_int_val, nullptr, bt->nz2, w.dWt, s, G->intent_b));
    } else {
        INTEL_TRY(dense_rows_linear_bwd(B * d->H2, I, dint, bt->his_item_int, w.e2.dseq + diid, d2, w.e2.nz_idx, w.e2.nz_val,
                                        w.e2.nz_cnt, NZ_CAP, w.dWt, s, G->intent_b));
    }
    return transpose(I, dint, w.dWt, G->intent_w, 1, s);
}

int intel_intent_bwd(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                     const float* d_intents, const float* d_intents_extra, intel_tensors_t* G, void* workspace,
                     size_t workspace_bytes, intel_stream_t stream) {
    return intel_intent_bwd_rows(d, P, bt, intents, d_intents, d_intents_extra, G, workspace, workspace_bytes, stream, nullptr);
}

}  // extern "C"
