// Internal (C++) launch interface between the orchestration code (api_*.cu) and the kernels.
// Everything is asynchronous on `s`; int return = INTEL_* status.
#pragma once
#include "common.cuh"
#include "intel_b200.h"   // parameter structs of the C ABI (intel_encoder_t) used by the fused encoder

namespace intel {

// ---- gemm.cu: fp32-parity (3xTF32) GEMM of the nn.Linear passes, C[M,N] = epilogue(A B^T) ----------------
// The pass fixes the operand layouts: FWD   A [M][K], B [N][K]  (Y = X W^T, linear)
//                                     DGRAD A [M][K], B [K][N]  (dX = dY W, linear_dx)
//                                     WGRAD A [K][M], B [K][N]  (dW += dY^T X, linear_dw; accumulate == 2, the inner
//                                                                dimension may be split over CTAs)
enum class GemmPass { FWD, DGRAD, WGRAD };
struct Gemm {
    GemmPass pass = GemmPass::FWD;
    int64_t M = 0, N = 0, K = 0;
    const float* A = nullptr; int64_t lda = 0;
    const float* B = nullptr; int64_t ldb = 0;
    float* C = nullptr; int64_t ldc = 0;
    const float* bias = nullptr;                        // + bias[n]
    const float* add = nullptr; int64_t ldadd = 0;      // + add[m,n]
    const float* mask = nullptr; int64_t ldmask = 0;    // *= (mask[m,n] > 0)   (relu backward)
    bool relu_a = false, relu_b = false, relu_out = false;
    int accumulate = 0;   // 0: C = r   1: C += r   2: atomicAdd(C, r)
    // optional list of the rows that matter (device int32 [*nrows], *nrows on the device too): the rows of A and C for a
    // forward / input-gradient product, the contracted rows for a weight gradient.  Rows that are not listed are padding
    // (history slots behind a session's length): the persistent tcgen05 kernels walk the list and never touch them, the
    // generic kernels ignore the list and compute them as well - the listed rows come out the same either way.  A weight
    // gradient on a generic kernel contracts the unlisted rows too: they must hold zeros unless gemm_rows_only(g).
    const int32_t* rows = nullptr;
    const int32_t* nrows = nullptr;
};
int gemm(const Gemm& g, cudaStream_t s);
void gemm_debug_use_tcgen05(int on);     // off: every product on the mma.sync kernels
void gemm_debug_use_rows_gemm(int on);   // off: not the two persistent kernels below (the generic tcgen05 kernel stays)
// launch status of a product, recorded by the profiler as gemm_fwd / gemm_dgrad / gemm_wgrad, and per shape as
// "<name>[MxNxK,<tag>]" under prof_detail(); tag_fmt is a printf format
int gemm_check_launch(const Gemm& g, const char* tag_fmt, ...);
// true when gemm(g) reads and writes the rows listed in g.rows alone (a persistent kernel below takes the product); rows
// outside the list then need not hold zeros
bool gemm_rows_only(const Gemm& g);
// gemm_rows_tc.cu: persistent tcgen05 kernel for tall products with a resident weight operand; false = shape not taken;
// status null: nothing is launched
bool gemm_rows_tc_try(const Gemm& g, cudaStream_t s, int* status);
// gemm_wgrad_tc.cu: dW += dY^T X over tens of thousands of rows, both operands MN-major natural tiles; same convention
bool gemm_wgrad_tc_try(const Gemm& g, cudaStream_t s, int* status);
// the products of linear_dx / linear_dw (below) as descriptors, for callers that ask gemm_rows_only first
Gemm dgrad_gemm(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* W, int64_t ldw, float* dX,
                int64_t lddx, const int32_t* rows, const int32_t* nrows);
Gemm wgrad_gemm(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW,
                int64_t lddw, const int32_t* rows, const int32_t* nrows);
// C[M,N] = A[M,K] W[N,K]^T (+bias)
int linear(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const float* W, int64_t ldw,
           const float* bias, float* C, int64_t ldc, cudaStream_t s, bool relu_a = false, bool relu_out = false,
           const float* add = nullptr, int64_t ldadd = 0, const int32_t* rows = nullptr, const int32_t* nrows = nullptr);
// dX[M,K] (=|+=) dY[M,N] W[N,K]  (optionally masked by relu input)
int linear_dx(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* W, int64_t ldw,
              float* dX, int64_t lddx, cudaStream_t s, int accumulate = 0, const float* mask = nullptr,
              int64_t ldmask = 0, const int32_t* rows = nullptr, const int32_t* nrows = nullptr);
// dW[N,K] += dY[M,N]^T X[M,K];  db[N] += colsum(dY)   (db may be null)
int linear_dw(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* X, int64_t ldx,
              float* dW, int64_t lddw, float* db, cudaStream_t s, bool relu_x = false, const int32_t* rows = nullptr,
              const int32_t* nrows = nullptr);
int colsum(int64_t M, int64_t N, const float* X, int64_t ld, float* out, cudaStream_t s);

// ---- embed.cu ---------------------------------------------------------------------------------
// table_rows > 0: ids outside [0, table_rows) read as a zero row / are skipped by the scatter (memory safety; the
// error itself is reported by batch_validate)
int gather_rows(int64_t rows, int d, const float* table, const int64_t* idx, float* out, int64_t ld_out,
                int relu, cudaStream_t s, int64_t table_rows = 0);
// grad_table[idx[r]] += d_out[r] (* (table[idx[r]] > 0) when relu_table != null); slot != null: the destination row is
// slot[idx[r]] (the compact gradient of a row set, sparse.cu)
int scatter_add_rows(int64_t rows, int d, const float* d_out, int64_t ld, const int64_t* idx, float* grad_table,
                     const float* relu_table, cudaStream_t s, int64_t table_rows = 0, const int32_t* slot = nullptr);
// ORs a bit into flags[0] for every class of out-of-range input (bit values: INTEL_BAD_* of intel_b200.h)
struct ValidateArgs {
    int64_t B, L, H1, H2, I, item_rows, class_rows, user_rows, ctx_rows;
    const int64_t *u_id, *i_id, *i_class, *session_len, *context_mh, *his_context, *history_len, *his_item_id, *history_item_len;
    const int32_t *idx1, *idx2;
    int nz1, nz2;
};
int batch_validate(const ValidateArgs& a, int32_t* flags, cudaStream_t s);

// Dense float64 rows X[R, I] times the intent_embeddings weight, exploiting that the rows are (nearly)
// one-hot / few-hot: Y[r, :] = sum_i float(X[r,i]) * Wt[i, :] + bias.  Wt is the [I, d] transpose.
// The non-zeros met on the way are compacted (cap entries per row) so the backward pass does not have
// to stream the dense rows again; rows with more than `cap` non-zeros are re-streamed.
int dense_rows_linear_fwd(int64_t R, int64_t I, int d, const double* X, const float* Wt, const float* bias,
                          float* Y, int64_t ldy, int32_t* nz_idx, float* nz_val, int32_t* nz_cnt, int cap,
                          cudaStream_t s, int64_t group = 0,
                          const int64_t* lens = nullptr);
// dWt[i, :] += float(X[r,i]) * dY[r, :]
int dense_rows_linear_bwd(int64_t R, int64_t I, int d, const double* X, const float* dY, int64_t lddy,
                          const int32_t* nz_idx, const float* nz_val, const int32_t* nz_cnt, int cap,
                          float* dWt, cudaStream_t s, float* db = nullptr);   // db (nullable): += column sums of dY (the bias gradient)
// compact rows: Y[r,:] = sum_e val[r,e] * Wt[idx[r,e],:] + bias.  Its backward is dense_rows_linear_bwd with
// X = null, nz_idx/nz_val = the caller's arrays, nz_cnt = null, cap = nz.
int sparse_rows_linear_fwd(int64_t R, int nz, int d, const int32_t* idx, const float* val, const float* Wt,
                           const float* bias, float* Y, int64_t ldy, cudaStream_t s);
// out[c, r] (=|+=) in[r, c]
int transpose(int64_t rows, int64_t cols, const float* in, float* out, int accumulate, cudaStream_t s);
// scores f64 [R,K] -> Y[R, d] = W[d,K] x + b  (score_embeddings) and the f32 copy xs[R,K]
int score_embed_fwd(int64_t R, int K, int d, const double* scores, const float* W, const float* b, float* Y,
                    float* xs, cudaStream_t s);
// backward of score_embeddings in one pass over dY: gW[d,K] += dY^T xs, gb[d] += column sums  (K <= 8, d <= 64)
bool score_embed_bwd_ok(int K, int d);
int score_embed_bwd(int64_t R, int K, int d, const float* dY, int64_t lddy, const float* xs, float* gW, float* gb,
                    cudaStream_t s);
// seq[b, t, :] += pos[(t < len[b]) ? t : 0, :]   (BERT4RecEncoder positions)
int add_positions(int64_t B, int64_t T, int d, const int64_t* lens, const float* pos, float* seq, cudaStream_t s);
// d_pos[(t < len[b]) ? t : 0, :] += d_seq[b, t, :]
int add_positions_bwd(int64_t B, int64_t T, int d, const int64_t* lens, const float* d_seq, float* d_pos,
                      cudaStream_t s);
// out[b, :] = X[b, len[b]-1, :]   and its backward (dX zero elsewhere; dX must be pre-zeroed)
int take_last(int64_t B, int64_t T, int d, const int64_t* lens, const float* X, float* out, int64_t ld_out,
              cudaStream_t s);
int take_last_bwd(int64_t B, int64_t T, int d, const int64_t* lens, const float* d_out, int64_t ld, float* dX,
                  cudaStream_t s);
int fill_zero(void* p, size_t bytes, cudaStream_t s);
int copy_d2d(void* dst, const void* src, size_t bytes, cudaStream_t s);

// ---- attn.cu ------------------------------------------------------------------------------------
// LayerNorm over the last dim (eps 1e-5); stats[r] = {mean, rstd}
int layernorm_fwd(int64_t R, int d, const float* Z, const float* gamma, const float* beta, float* Y,
                  float* stats, cudaStream_t s);
int layernorm_bwd(int64_t R, int d, const float* dY, const float* Z, const float* stats, const float* gamma,
                  float* dZ, float* dgamma, float* dbeta, cudaStream_t s);
// Multi-head attention without output projection (layers.py:31-60).  QKV [B,T,3d] (q|k|v), O [B,T,d].
// lens == null: every slot is a live key (IntEL stacks); else keys j >= lens[b] are masked (BERT4Rec).
int mha_fwd(int64_t B, int64_t T, int d, int heads, const float* QKV, const int64_t* lens, float* O,
            cudaStream_t s);
int mha_bwd(int64_t B, int64_t T, int d, int heads, const float* QKV, const int64_t* lens, const float* dO,
            float* dQKV, cudaStream_t s);
// Pooled cross attention (attention.py:54-63 collapsed, SURVEY 8a-4): att_j = scale * X[b,j].qk[b],
// shift by the max over all L slots, softmax over j < n_b, xbar = sum_j p_j X[b,j].
// width-32 streams: the pooling with q -> qk = W_k^T q in front and xbar -> W_v xbar behind it in one kernel; the backward
// kernel returns d(q) and accumulates d(W_k), d(W_v)
bool cross_full_ok(int d, int64_t L);
int cross_full_fwd(int64_t B, int64_t L, const float* X, const float* q, int64_t ldq, const float* Wk, const float* Wv,
                   const int64_t* lens, float scale, float* p, float* qk_out, float* xbar_out, float* out, int64_t ldo, cudaStream_t s);
int cross_full_bwd(int64_t B, int64_t L, const float* X, const float* q, int64_t ldq, const float* qk, const float* Wk, const float* Wv,
                   const int64_t* lens, float scale, const float* p, const float* xbar, const float* dout, int64_t ldd, float* dX,
                   float* dq_out, int64_t lddq, float* gWk, float* gWv, cudaStream_t s);
int cross_pool_fwd(int64_t B, int64_t L, int d, const float* X, const float* qk, const int64_t* lens,
                   float scale, float* p, float* xbar, cudaStream_t s);
// dX[b,j] (=) p_j dxbar + scale datt_j qk ; dqk[b] = scale sum_j datt_j X[b,j]
int cross_pool_bwd(int64_t B, int64_t L, int d, const float* X, const float* qk, const int64_t* lens,
                   float scale, const float* p, const float* dxbar, float* dX, float* dqk, cudaStream_t s);
// softmax over rows and its backward: dZ = p * (dP - sum(p dP))
int softmax_rows(int64_t R, int64_t N, const float* Z, float* P, cudaStream_t s, int64_t ldz = 0);   // ldz: row stride of Z (0 = N)
int softmax_rows_bwd(int64_t R, int64_t N, const float* P, const float* dP, const float* dP2, float* dZ,
                     cudaStream_t s, int64_t ldz = 0);   // incoming gradient dP + dP2 (dP2 nullable)

// ---- bert_fused.cu: BERT4RecEncoder forward in one kernel (d = 32, T <= 24, 1 or 2 heads) -------------------------------
bool bert_fused_ok(int64_t T, int d, int heads, int layers);
void bert_debug_use_fused(int on);
// seq [B,T,32]: token embeddings in; with save it receives X[0] (positions added) and the per-layer activations of bert_bwd
// are written (QKV [B*T,96], Z1, C, F, Z2, X[l+1] [B*T,32], st1 / st2 [B*T,2]); out[b, :] = state at len - 1
int bert_fused_fwd(int64_t B, int64_t T, int heads, int layers, const int64_t* lens, const intel_encoder_t& p, float* seq,
                   float* const* X, float* const* QKV, float* const* Z1, float* const* st1, float* const* C, float* const* F,
                   float* const* Z2, float* const* st2, bool save, float* out, int64_t ld_out, cudaStream_t s);

// ---- gru.cu -------------------------------------------------------------------------------------
// GRU recurrence for hidden size 128 (gate order r,z,n; torch.nn.GRU equations): one CTA per tile of sessions walks all T
// steps with W_hh resident in shared memory (see gru.cu).  gi [B,T,3h] (input projections incl. b_ih), h_all [B,T+1,h]
// (slot 0 pre-zeroed), gates [B,T,4h] = (r, z, n, gh_n), dgi [B,T,3h], dgh_all [B,T+1,3h] (slot T pre-zeroed),
// dh_in [B,h] = d loss / d h_T.
int gru_seq_fwd(int64_t B, int64_t T, const int64_t* lens, const float* gi, const float* w_hh, const float* b_hh, float* h_all,
                float* gates, cudaStream_t s);
// tcgen05 forward recurrence (gru_tc.cu) of up to two encoders in one launch: clusters of four CTAs, W_hh slices resident as
// UMMA B operands; same outputs.  order (nullable): sessions by decreasing length (gru_prep)
struct GruTcOne {
    int64_t B, T;
    const int64_t* lens;
    const float *gi, *w_hh, *b_hh;
    float *h_all, *gates;
    const int32_t* order;
};
struct GruTcPair { GruTcOne e[2]; int n, save_gates; };    // save_gates = 0: forward only, gates are not written
bool gru_tc_supported();
int gru_tc_fwd_pair(const GruTcPair& p, cudaStream_t s);
void gru_debug_use_tcgen05(int on);
// backward recurrence of up to two encoders in one launch.  order (nullable): sessions by decreasing length (gru_prep);
// counter (nullable; needed for two encoders): the encoder's tile counter, zero on entry (tiles round robin without it).
// live_only: dgi / dgh_all rows of padding slots (t >= len) are left unwritten, for products that read the live rows
// alone; otherwise they are written as zeros, except slot T of dgh_all, which the caller clears
struct GruBwdOne {
    int64_t B, T;
    const int64_t* lens;
    const float *w_hh, *h_all, *gates, *dh_in;
    float *dgi, *dgh_all, *db_ih, *db_hh;
    const int32_t* order;
    int32_t* counter;
    int live_only;
};
struct GruBwdPair { GruBwdOne e[2]; int n; };
int gru_seq_bwd_pair(const GruBwdPair& p, cudaStream_t s);
// output projections (Linear(128 -> d <= 64), no bias) of both encoders in one launch, and their input gradients
bool gru_outproj_pair_ok(int n0, int n1);
int gru_outproj_pair_fwd(int64_t B, const int* n, const float* const* W, const float* const* h_last, const int64_t* ldh,
                         float* const* out, const int64_t* ldo, cudaStream_t s);
int gru_outproj_pair_dx(int64_t B, const int* n, const float* const* W, const float* const* dout, const int64_t* ldd,
                        float* const* dh, const int64_t* ldh, cudaStream_t s);
// For up to two encoders in one launch, one entry each (null pointers skip a part):
// - the live (session, step) pairs of a padded [B, T] history as row numbers, in (b, t) order: rows_t[i] = b T + t into the
//   [B, T, .] tensors, rows_t1[i] = b (T + 1) + t into the [B, T + 1, .] ones; *count = sum of the (clamped) lengths;
// - order [B + 1]: order[i] = session with the i-th longest history (stable; T <= 63), order[B] = 0 (the tile counter).  With
//   it the backward recurrence walks tiles of equally long sessions and stops each tile at its own last step (the reference
//   packs the sequences: GeneralSeq.py:64-71).
struct GruPrepOne { int64_t B; int T; const int64_t* lens; int32_t *rows_t, *rows_t1, *count, *order; };
int gru_prep(int n, const GruPrepOne* e, cudaStream_t s);

// ---- trunk.cu: fused self-attention stack (d = 32, L <= 64): all layers of a session on chip -----
// The activations of one self-attention stack (IntEL.py:182-197) over R = B*L rows of width d, as the forward pass leaves
// them for the backward pass: X[0] = input, X[l+1] = output of layer l (layers <= 8); per layer q|k|v [R,3d], attention
// output, FFN hidden (pre-relu), pre-LN sum [R,d] each, LN mean / rstd [R,2].  The fused and the staged paths read them alike.
struct StackWs {
    float* X[9];
    float* QKV[8];
    float* A[8];
    float* U[8];
    float* Z[8];
    float* st[8];
};
inline void stack_layout(Arena& a, int64_t R, int d, int layers, StackWs& w) {
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
int adam_step(int count, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
              const int64_t* numel, const float* weight_decay, double lr, double beta1, double beta2, double eps, int64_t step,
              cudaStream_t s);
int pool_head_fwd(int64_t B, int64_t L, int K, const float* Wl, const double* scores, float* weights, float* ens, float* p,
                  float* w, cudaStream_t s);
int pool_head_bwd(int64_t B, int64_t L, int K, const double* scores, const float* p, const float* w, const float* d_weights,
                  const float* d_ens, float* dWl, cudaStream_t s);
int awelv_fwd(int64_t B, int64_t L, int K, int h, const float* U, const float* M, const int64_t* uid, const double* scores,
              float* weights, float* ens, float* wsmall, cudaStream_t s);
int awelv_bwd(int64_t B, int64_t L, int K, int h, const float* U, const float* M, const int64_t* uid, const double* scores,
              const float* wsmall, const float* d_weights, const float* d_ens, float* gU, float* gM, cudaStream_t s);
static const int TD = 32;            // stream width of the fused stack kernels
struct TrunkArgs {
    int64_t B;
    int L, heads, layers;
    const float *wq, *wk, *wv, *w1, *b1, *w2, *b2, *lnw, *lnb;
    float* X[9];                     // X[0] input, X[l+1] output of layer l, each [B*L, 32]
    // activations of layer l kept for the backward pass (written by the forward kernel when save != 0):
    float *QKV[8], *A[8], *U[8], *Z[8], *ST[8];   // [B*L,96] q|k|v, [B*L,32] x3, [B*L,2] LN mean / rstd
    int save;
    Dropout drop[8];                 // per layer (p = 0: off)
    // backward only
    float* dX;                       // [B*L,32]: d loss / d X[layers] on entry, d loss / d X[0] on return
    float *gwq, *gwk, *gwv, *gw1, *gb1, *gw2, *gb2, *glnw, *glnb;
};
// tcgen05 / tensor-memory forward pass of the same stack (trunk_tc.cu): L <= 128, same saved activations
bool trunk_tc_supported(const TrunkArgs& a);
int trunk_tc_fwd(const TrunkArgs& a, cudaStream_t s);
void trunk_debug_use_tcgen05(int on);
void trunk_debug_sessions_per_cta(int n);
void trunk_reserve_sms(int n);      // SMs the persistent backward kernel leaves to a concurrent collective ...
void trunk_reserve_apply(bool on);  // ... in the launches made while this is on
bool trunk_supported(int64_t L, int d, int heads, int layers);      // mma.sync kernels, forward and backward
bool trunk_fwd_supported(int64_t L, int heads, int layers);         // any fused forward kernel (d = 32)
// w.X[0] = stack input [B*L,32]; w.X[l+1] receives the output of layer l
int trunk_fwd(int64_t B, int64_t L, int heads, int layers, const intel_selfatt_t& p, const StackWs& w, float drop_p,
              uint64_t drop_seed, int stream_id, cudaStream_t s, bool save = true);
// dX: d loss / d X[layers] on entry, d loss / d X[0] on return; weight gradients are accumulated into g
int trunk_bwd(int64_t B, int64_t L, int heads, int layers, const intel_selfatt_t& p, const intel_selfatt_t& g, const StackWs& w,
              float* dX, float drop_p, uint64_t drop_seed, int stream_id, cudaStream_t s);

// ---- fuse.cu ------------------------------------------------------------------------------------
// weights[b,l,:] = l < n_b ? w_valid[b] : w_pad[b];  ens[b,l] = sum_k weights * float(scores)
int head_fuse_fwd(int64_t B, int64_t L, int K, const float* w_valid, const float* w_pad, const double* scores,
                  const int64_t* lens, float* weights, float* ens, cudaStream_t s);
// dw_valid[b,k] = sum_{l<n} g, dw_pad[b,k] = sum_{l>=n} g with g = d_weights[b,l,k] + d_ens[b,l] x[b,l,k]
int head_fuse_bwd(int64_t B, int64_t L, int K, const float* d_weights, const float* d_ens, const double* scores,
                  const int64_t* lens, float* dw_valid, float* dw_pad, cudaStream_t s);
// the head's nn.Linear(D, K) folded into the two kernels above (K = 2..4, D <= 256): all [B, D] = head input of the valid rows,
// pad rows see the inputs >= off_u only; the backward call writes d(all) [B, D] and accumulates the head's weight / bias gradient
bool head_full_ok(int K, int D);
int head_full_fwd(int64_t B, int64_t L, int K, int D, int off_u, const float* all, const float* Wh, const float* bh,
                  const double* scores, const int64_t* lens, float* weights, float* ens, cudaStream_t s);
int head_full_bwd(int64_t B, int64_t L, int K, int D, int off_u, const float* all, const float* Wh, const float* d_weights,
                  const float* d_ens, const double* scores, const int64_t* lens, float* dall, float* gWh, float* gbh, cudaStream_t s);
// per-item variant (cross_attention = 0): ens[b,l] = sum_k weights[b,l,k] x ; g[b,l,k] as above
int item_fuse_fwd(int64_t R, int K, const float* weights, const double* scores, float* ens, cudaStream_t s);
int item_fuse_bwd(int64_t R, int K, const float* d_weights, const float* d_ens, const double* scores, float* g,
                  cudaStream_t s);
// gate (cross_attention = 0): Y[b,l,:] = X[b,l,:] * m[b,:]  and backward
int gate_fwd(int64_t B, int64_t L, int d, const float* X, const float* m, float* Y, int64_t ldy, cudaStream_t s);
int gate_bwd(int64_t B, int64_t L, int d, const float* X, const float* m, const float* dY, int64_t lddy,
             float* dX, float* dm, cudaStream_t s);
// out[b,l,:] = v[b,:] broadcast into a strided slice; and the reduction sum_l back
int bcast_rows(int64_t B, int64_t L, int d, const float* v, int64_t ldv, float* out, int64_t ldo, cudaStream_t s);
int bcast_rows_bwd(int64_t B, int64_t L, int d, const float* dout, int64_t ldo, float* dv, int64_t ldv,
                   int accumulate, cudaStream_t s);
// y = x * (v > 0)
int relu_bwd(int64_t rows, int cols, const float* dy, int64_t lddy, const float* v, int64_t ldv, float* dx,
             int64_t lddx, cudaStream_t s);
int add_inplace(int64_t n, float* y, const float* x, cudaStream_t s);
// y = relu(x + b) on strided row views (b nullable)
int bias_relu_rows(int64_t rows, int cols, const float* x, int64_t ldx, const float* b, float* y, int64_t ldy, cudaStream_t s);
// y = x * dropout mask/(1-p) (+ add); used by the staged path of the stacks, forward and backward
int dropout_apply(int64_t rows, int width, const float* x, const float* add, float* y, const Dropout& dr, cudaStream_t s);

}  // namespace intel
