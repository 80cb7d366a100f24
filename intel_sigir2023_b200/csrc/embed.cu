// Embedding gathers / dense-gradient scatter-adds, the dense-row intent embedding, and small
// layout kernels.  All HBM-bound: coalesced / 16-byte vector accesses, grids sized to the SM count.
#include "kernels.h"

namespace intel {

// ------------------------------------------------------------------------------------------------
// gather: out[r, 0:d] = table[idx[r], 0:d]   (nn.Embedding forward; IntEL.py:135,141,147,148,170,172,178)
// One thread per 16-byte chunk of an output row; rows of 16/32 floats are 64/128-byte segments.
template <int VEC>
__global__ void __launch_bounds__(256) gather_kernel(int64_t rows, int d, const float* __restrict__ table,
                                                     const int64_t* __restrict__ idx, float* __restrict__ out,
                                                     int64_t ld_out, int relu, int64_t table_rows) {
    const int per_row = d / VEC;
    const int64_t total = rows * per_row;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / per_row;
        const int c = (int)(e % per_row) * VEC;
        const int64_t id = idx[r];
        // an id outside the table (nn.Embedding raises IndexError; intel_batch_validate reports it) reads as a zero row
        const bool ok = table_rows <= 0 || (id >= 0 && id < table_rows);
        if (VEC == 4) {
            float4 v = ok ? *reinterpret_cast<const float4*>(table + id * d + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            *reinterpret_cast<float4*>(out + r * ld_out + c) = v;
        } else {
            float v = ok ? table[id * d + c] : 0.f;
            out[r * ld_out + c] = relu ? fmaxf(v, 0.f) : v;
        }
    }
}

int gather_rows(int64_t rows, int d, const float* table, const int64_t* idx, float* out, int64_t ld_out, int relu,
                cudaStream_t s, int64_t table_rows) {
    if (rows <= 0 || d <= 0) return INTEL_OK;
    INTEL_REQUIRE(table && idx && out, INTEL_ERR_ARG, "gather: null pointer");
    const bool vec = (d % 4 == 0) && (ld_out % 4 == 0) && (((uintptr_t)table | (uintptr_t)out) % 16 == 0);
    const int64_t total = rows * (vec ? d / 4 : d);
    unsigned grid = stream_grid(ceil_div(total, 256), 8);
    if (vec) { auto k = gather_kernel<4>; LAUNCH(k, dim3(grid), dim3(256), 0, s, rows, d, table, idx, out, ld_out, relu, table_rows); }
    else { auto k = gather_kernel<1>; LAUNCH(k, dim3(grid), dim3(256), 0, s, rows, d, table, idx, out, ld_out, relu, table_rows); }
    return check_launch("gather", (double)rows * (8.0 * d + 8.0), 0.0);
}

// scatter-add: grad_table[idx[r], :] += d_out[r, :]   (embedding_dense_backward; the gradient stays
// DENSE so torch.optim.Adam(weight_decay) is a drop-in).  fp32 atomics.
// REMAP (sparse table gradients, sparse.cu): the destination row is slot[idx[r]], a row of the compact [U, d] gradient of
// the step's row set; the ReLU gate still reads the parameter row of the original id.
template <bool REMAP>
__global__ void __launch_bounds__(256) scatter_add_kernel(int64_t rows, int d, const float* __restrict__ d_out,
                                                          int64_t ld, const int64_t* __restrict__ idx,
                                                          float* grad_table, const float* __restrict__ relu_table,
                                                          int64_t table_rows, const int32_t* __restrict__ slot) {
    const int64_t total = rows * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / d;
        const int c = (int)(e % d);
        const int64_t id = idx[r];
        if (table_rows > 0 && (id < 0 || id >= table_rows)) continue;      // would land in another parameter's gradient
        float g = d_out[r * ld + c];
        if (relu_table && !(relu_table[id * d + c] > 0.f)) g = 0.f;
        const int64_t dst = REMAP ? (int64_t)slot[id] : id;
        if (g != 0.f) atomicAdd(grad_table + dst * d + c, g);
    }
}

int scatter_add_rows(int64_t rows, int d, const float* d_out, int64_t ld, const int64_t* idx, float* grad_table,
                     const float* relu_table, cudaStream_t s, int64_t table_rows, const int32_t* slot) {
    if (rows <= 0 || d <= 0) return INTEL_OK;
    INTEL_REQUIRE(d_out && idx && grad_table, INTEL_ERR_ARG, "scatter_add: null pointer");
    INTEL_REQUIRE(!slot || table_rows > 0, INTEL_ERR_ARG, "scatter_add: a row-slot map needs the table's row count");
    unsigned grid = stream_grid(ceil_div(rows * d, 256), 8);
    if (slot) {
        auto k = scatter_add_kernel<true>;
        LAUNCH(k, dim3(grid), dim3(256), 0, s, rows, d, d_out, ld, idx, grad_table, relu_table, table_rows, slot);
    } else {
        auto k = scatter_add_kernel<false>;
        LAUNCH(k, dim3(grid), dim3(256), 0, s, rows, d, d_out, ld, idx, grad_table, relu_table, table_rows, slot);
    }
    return check_launch("scatter_add", (double)rows * (12.0 * d + 8.0), (double)rows * d);
}

// ------------------------------------------------------------------------------------------------
// Range check of every index a batch feeds to the tables (nn.Embedding raises IndexError on these, IntEL.py:135-178)
// and of the history lengths the encoders index with (pack_padded_sequence / the last-state gather need 1..H).
// One pass over the int64 fields, a few KB per session; bits are ORed into flags[0].
__device__ __forceinline__ void check_ids(const int64_t* v, int64_t n, int64_t lo, int64_t hi, int bit, int& bad) {
    if (!v) return;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t x = v[e];
        if (x < lo || x >= hi) bad |= bit;
    }
}
__global__ void __launch_bounds__(256) batch_validate_kernel(ValidateArgs a, int32_t* flags) {
    int bad = 0;
    check_ids(a.u_id, a.B, 0, a.user_rows, 1, bad);
    check_ids(a.i_id, a.B * a.L, 0, a.item_rows, 2, bad);
    if (a.class_rows > 0) check_ids(a.i_class, a.B * a.L, 0, a.class_rows, 4, bad);
    check_ids(a.context_mh, a.B, 0, a.ctx_rows, 8, bad);
    check_ids(a.his_context, a.B * a.H1, 0, a.ctx_rows, 8, bad);
    check_ids(a.his_item_id, a.B * a.H2, 0, a.item_rows, 2, bad);
    check_ids(a.session_len, a.B, 0, a.L + 1, 16, bad);
    check_ids(a.history_len, a.B, 1, a.H1 + 1, 32, bad);
    check_ids(a.history_item_len, a.B, 1, a.H2 + 1, 32, bad);
    if (a.idx1)
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < a.B * a.H1 * a.nz1; e += (int64_t)gridDim.x * blockDim.x)
            if (a.idx1[e] < 0 || a.idx1[e] >= a.I) bad |= 64;
    if (a.idx2)
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < a.B * a.H2 * a.nz2; e += (int64_t)gridDim.x * blockDim.x)
            if (a.idx2[e] < 0 || a.idx2[e] >= a.I) bad |= 64;
    if (bad) atomicOr(flags, bad);
}
int batch_validate(const ValidateArgs& a, int32_t* flags, cudaStream_t s) {
    INTEL_REQUIRE(flags, INTEL_ERR_ARG, "batch_validate: null flag pointer");
    if (a.B <= 0) return INTEL_OK;
    const unsigned grid = stream_grid(ceil_div(a.B * (a.L > a.H1 ? a.L : a.H1), 256), 4);
    LAUNCH(batch_validate_kernel, dim3(grid), dim3(256), 0, s, a, flags);
    return check_launch("batch_validate", 8.0 * (double)a.B * (2.0 * a.L + a.H1 + a.H2 + 6.0), 0.0);
}

// ------------------------------------------------------------------------------------------------
// Dense float64 rows -> intent embedding (IntEL.py:136,142: nn.Linear(I, d_int) applied to the dense
// [B,H,I] his_intents / one-hot his_item_int).  These two tensors are ~93% of the batch bytes
// (SURVEY.md 8a-1), so the kernel is a pure HBM stream: one warp per row, 8-byte coalesced loads with
// 4 loads in flight per lane, and arithmetic only for the (few) non-zero entries met on the way.
static const int DR_UNROLL = 4;

__device__ __forceinline__ void dense_row_accumulate(const double* __restrict__ x, int64_t I, int d, int lane,
                                                     const float* __restrict__ Wt, float& acc0, float& acc1,
                                                     int32_t* nz_idx, float* nz_val, int cap, int& cnt) {
    for (int64_t base = 0; base < I; base += 32 * DR_UNROLL) {
        double v[DR_UNROLL];
#pragma unroll
        for (int u = 0; u < DR_UNROLL; ++u) {
            int64_t i = base + u * 32 + lane;
            v[u] = (i < I) ? x[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < DR_UNROLL; ++u) {
            unsigned m = __ballot_sync(0xffffffffu, v[u] != 0.0);
            while (m) {
                const int src = __ffs((int)m) - 1;
                m &= m - 1;
                const float fv = (float)__shfl_sync(0xffffffffu, v[u], src);
                const int64_t i = base + u * 32 + src;
                if (Wt) {
                    if (lane < d) acc0 = fmaf(fv, Wt[i * d + lane], acc0);
                    if (lane + 32 < d) acc1 = fmaf(fv, Wt[i * d + lane + 32], acc1);
                }
                if (nz_idx && lane == 0 && cnt < cap) { nz_idx[cnt] = (int32_t)i; nz_val[cnt] = fv; }
                cnt++;
            }
        }
    }
}

__global__ void __launch_bounds__(256) dense_rows_fwd_kernel(int64_t R, int64_t I, int d, const double* __restrict__ X,
                                                             const float* __restrict__ Wt, const float* __restrict__ bias,
                                                             float* __restrict__ Y, int64_t ldy, int32_t* nz_idx,
                                                             float* nz_val, int32_t* nz_cnt, int cap, int64_t group,
                                                             const int64_t* __restrict__ lens) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < R; r += nwarps) {
        float acc0 = (bias && lane < d) ? bias[lane] : 0.f;
        float acc1 = (bias && lane + 32 < d) ? bias[lane + 32] : 0.f;
        int cnt = 0;
        // padding rows behind a session's history length are zeros by construction (collate_batch) and never read by the
        // encoders: their output is the bias, without streaming 8 I bytes of zeros
        const bool pad = lens != nullptr && (r % group) >= lens[r / group];
        if (!pad)
            dense_row_accumulate(X + r * I, I, d, lane, Wt, acc0, acc1, nz_idx ? nz_idx + r * cap : nullptr,
                                 nz_val ? nz_val + r * cap : nullptr, cap, cnt);
        if (lane < d) Y[r * ldy + lane] = acc0;
        if (lane + 32 < d) Y[r * ldy + lane + 32] = acc1;
        if (nz_cnt && lane == 0) nz_cnt[r] = cnt;
    }
}

int dense_rows_linear_fwd(int64_t R, int64_t I, int d, const double* X, const float* Wt, const float* bias, float* Y,
                          int64_t ldy, int32_t* nz_idx, float* nz_val, int32_t* nz_cnt, int cap, cudaStream_t s, int64_t group,
                          const int64_t* lens) {
    if (R <= 0) return INTEL_OK;
    INTEL_REQUIRE(d <= 64, INTEL_ERR_UNSUPPORTED, "intent_emb_size %d > 64 not supported", d);
    INTEL_REQUIRE(X && Wt && Y, INTEL_ERR_ARG, "dense_rows_linear_fwd: null pointer");
    unsigned grid = stream_grid(ceil_div(R, 8), 8);
    if (group <= 0) lens = nullptr;
    // ragged input: one warp per row and no grid-stride loop, so that the block scheduler balances live and padding rows
    if (lens) grid = (unsigned)ceil_div(R, 8);
    LAUNCH(dense_rows_fwd_kernel, dim3(grid), dim3(256), 0, s, R, I, d, X, Wt, bias, Y, ldy, nz_idx, nz_val, nz_cnt, cap,
           group > 0 ? group : 1, lens);
    return check_launch("dense_rows_fwd", (double)R * (8.0 * I + 4.0 * d), 0.0);
}

// Compact input form of the same layer: row r = sum_e val[r,e] * Wt[idx[r,e], :] + bias (one thread per output).
__global__ void __launch_bounds__(256) sparse_rows_fwd_kernel(int64_t R, int nz, int d, const int32_t* __restrict__ idx,
                                                              const float* __restrict__ val, const float* __restrict__ Wt,
                                                              const float* __restrict__ bias, float* __restrict__ Y,
                                                              int64_t ldy) {
    const int64_t total = R * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / d;
        const int c = (int)(e % d);
        float acc = bias ? bias[c] : 0.f;
        for (int k = 0; k < nz; ++k) {
            const float v = val[r * nz + k];
            if (v != 0.f) acc = fmaf(v, Wt[(int64_t)idx[r * nz + k] * d + c], acc);
        }
        Y[r * ldy + c] = acc;
    }
}

int sparse_rows_linear_fwd(int64_t R, int nz, int d, const int32_t* idx, const float* val, const float* Wt,
                           const float* bias, float* Y, int64_t ldy, cudaStream_t s) {
    if (R <= 0) return INTEL_OK;
    INTEL_REQUIRE(idx && val && Wt && Y && nz > 0, INTEL_ERR_ARG, "sparse_rows_linear_fwd: bad argument");
    unsigned grid = stream_grid(ceil_div(R * d, 256), 8);
    LAUNCH(sparse_rows_fwd_kernel, dim3(grid), dim3(256), 0, s, R, nz, d, idx, val, Wt, bias, Y, ldy);
    return check_launch("sparse_rows_fwd", (double)R * (8.0 * nz + 4.0 * d * (nz + 1)), 2.0 * R * nz * d);
}

// backward w.r.t. the weight: dWt[i, :] += x[r,i] * dY[r, :]; uses the compacted non-zeros of the
// forward pass, re-streaming only rows that overflowed the compaction capacity.
__global__ void __launch_bounds__(256) dense_rows_bwd_kernel(int64_t R, int64_t I, int d, const double* __restrict__ X,
                                                             const float* __restrict__ dY, int64_t lddy,
                                                             const int32_t* __restrict__ nz_idx,
                                                             const float* __restrict__ nz_val,
                                                             const int32_t* __restrict__ nz_cnt, int cap, float* dWt, float* db) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float b0 = 0.f, b1 = 0.f;                  // column sums of dY over this warp's rows = its share of the bias gradient
    for (int64_t r = warp; r < R; r += nwarps) {
        const float g0 = (lane < d) ? dY[r * lddy + lane] : 0.f;
        const float g1 = (lane + 32 < d) ? dY[r * lddy + lane + 32] : 0.f;
        b0 += g0;
        b1 += g1;
        const int cnt = nz_cnt ? nz_cnt[r] : (X ? cap + 1 : cap);     // X == null: caller-provided compact rows
        if (cnt <= cap) {
            for (int e = 0; e < cnt; ++e) {
                const int64_t i = nz_idx[r * cap + e];
                const float fv = nz_val[r * cap + e];
                if (fv == 0.f) continue;
                if (lane < d) atomicAdd(dWt + i * d + lane, fv * g0);
                if (lane + 32 < d) atomicAdd(dWt + i * d + lane + 32, fv * g1);
            }
        } else {
            const double* x = X + r * I;
            for (int64_t base = 0; base < I; base += 32) {
                const int64_t ii = base + lane;
                const double v = (ii < I) ? x[ii] : 0.0;
                unsigned m = __ballot_sync(0xffffffffu, v != 0.0);
                while (m) {
                    const int src = __ffs((int)m) - 1;
                    m &= m - 1;
                    const float fv = (float)__shfl_sync(0xffffffffu, v, src);
                    const int64_t i = base + src;
                    if (lane < d) atomicAdd(dWt + i * d + lane, fv * g0);
                    if (lane + 32 < d) atomicAdd(dWt + i * d + lane + 32, fv * g1);
                }
            }
        }
    }
    if (db) {                                  // CTA-level sum first: one atomic per column and CTA
        __shared__ float red[8][64];
        const int wib = threadIdx.x >> 5;
        red[wib][lane] = b0;
        red[wib][lane + 32] = b1;
        __syncthreads();
        if (threadIdx.x < 64 && (int)threadIdx.x < d) {
            float t = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) t += red[q][threadIdx.x];
            if (t != 0.f) atomicAdd(db + threadIdx.x, t);
        }
    }
}

int dense_rows_linear_bwd(int64_t R, int64_t I, int d, const double* X, const float* dY, int64_t lddy,
                          const int32_t* nz_idx, const float* nz_val, const int32_t* nz_cnt, int cap, float* dWt,
                          cudaStream_t s, float* db) {
    if (R <= 0) return INTEL_OK;
    INTEL_REQUIRE(d <= 64, INTEL_ERR_UNSUPPORTED, "intent_emb_size %d > 64 not supported", d);
    unsigned grid = stream_grid(ceil_div(R, 8), 8);
    LAUNCH(dense_rows_bwd_kernel, dim3(grid), dim3(256), 0, s, R, I, d, X, dY, lddy, nz_idx, nz_val, nz_cnt, cap, dWt, db);
    return check_launch("dense_rows_bwd", (double)R * (4.0 * d + 4.0), 0.0);
}

// ------------------------------------------------------------------------------------------------
// out[c, r] (=|+=) in[r, c]  - 32x32 shared-memory tile transpose
__global__ void __launch_bounds__(256) transpose_kernel(int64_t rows, int64_t cols, const float* __restrict__ in,
                                                        float* out, int accumulate) {
    __shared__ float tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
    for (int i = ty; i < 32; i += 8) {
        int64_t r = r0 + i, c = c0 + tx;
        tile[i][tx] = (r < rows && c < cols) ? in[r * cols + c] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        int64_t c = c0 + i, r = r0 + tx;
        if (c < cols && r < rows) {
            float v = tile[tx][i];
            if (accumulate) out[c * rows + r] += v; else out[c * rows + r] = v;
        }
    }
}

int transpose(int64_t rows, int64_t cols, const float* in, float* out, int accumulate, cudaStream_t s) {
    if (rows <= 0 || cols <= 0) return INTEL_OK;
    dim3 grid((unsigned)ceil_div(cols, 32), (unsigned)ceil_div(rows, 32));
    LAUNCH(transpose_kernel, grid, dim3(256), 0, s, rows, cols, in, out, accumulate);
    return check_launch("transpose");
}

// ------------------------------------------------------------------------------------------------
// score_embeddings (IntEL.py:190): Y[r, c] = b[c] + sum_k W[c,k] float(scores[r,k]); xs = float(scores)
__global__ void __launch_bounds__(256) score_embed_kernel(int64_t R, int K, int d, const double* __restrict__ scores,
                                                          const float* __restrict__ W, const float* __restrict__ b,
                                                          float* __restrict__ Y, float* __restrict__ xs) {
    const int64_t total = R * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / d;
        const int c = (int)(e % d);
        float acc = b[c];
        for (int k = 0; k < K; ++k) acc = fmaf(W[c * K + k], (float)scores[r * K + k], acc);
        Y[e] = acc;
        if (xs && c < K) xs[r * K + c] = (float)scores[r * K + c];
    }
}

// Same, four output channels per thread: the thread's channel group is fixed (the grid stride is a multiple of d/4), so
// its 4 x K weights and biases stay in registers and every row costs K loads and one 16-byte store.
constexpr int SE_K = 8;
__global__ void __launch_bounds__(256) score_embed_v4_kernel(int64_t R, int K, int d, const double* __restrict__ scores,
                                                             const float* __restrict__ W, const float* __restrict__ b,
                                                             float* __restrict__ Y, float* __restrict__ xs) {
    const int gpr = d >> 2;                                    // channel groups per row
    const int cg = (int)(threadIdx.x % gpr);
    float wr[4][SE_K], br[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        br[j] = b[cg * 4 + j];
#pragma unroll
        for (int k = 0; k < SE_K; ++k) wr[j][k] = (k < K) ? W[(cg * 4 + j) * K + k] : 0.f;
    }
    const int64_t rpb = blockDim.x / gpr;                      // rows one CTA covers per sweep
    const int64_t r0 = (int64_t)blockIdx.x * rpb + threadIdx.x / gpr;
    const int64_t stride = (int64_t)gridDim.x * rpb;
    constexpr int UR = 1;                                      // rows in flight per thread (2 measured slower on the B200: 101
                                                               // registers, 29 us against 23 us per launch)
    for (int64_t rb = r0; rb < R; rb += UR * stride) {
        float x[UR][SE_K];
#pragma unroll
        for (int u = 0; u < UR; ++u) {
            const int64_t r = rb + u * stride;
#pragma unroll
            for (int k = 0; k < SE_K; ++k) x[u][k] = (k < K && r < R) ? (float)scores[r * K + k] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < UR; ++u) {
            const int64_t r = rb + u * stride;
            if (r >= R) break;
            float4 y;
            float* yy = &y.x;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float acc = br[j];
#pragma unroll
                for (int k = 0; k < SE_K; ++k)
                    if (k < K) acc = fmaf(wr[j][k], x[u][k], acc);
                yy[j] = acc;
            }
            *reinterpret_cast<float4*>(Y + r * d + cg * 4) = y;
            if (xs) {
#pragma unroll
                for (int k = 0; k < SE_K; ++k)
                    if (k < K && (k >> 2) == cg) xs[r * K + k] = x[u][k];
            }
        }
    }
}

int score_embed_fwd(int64_t R, int K, int d, const double* scores, const float* W, const float* b, float* Y, float* xs,
                    cudaStream_t s) {
    if (R <= 0) return INTEL_OK;
    INTEL_REQUIRE(!xs || K <= d, INTEL_ERR_UNSUPPORTED, "score_embed: model_num %d > s_emb_size %d", K, d);
    if (K <= SE_K && d % 4 == 0 && 256 % (d / 4) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0) {
        unsigned grid = stream_grid(ceil_div(R * (d / 4), 256 * 4), 8);
        LAUNCH(score_embed_v4_kernel, dim3(grid), dim3(256), 0, s, R, K, d, scores, W, b, Y, xs);
    } else {
        unsigned grid = stream_grid(ceil_div(R * d, 256), 8);
        LAUNCH(score_embed_kernel, dim3(grid), dim3(256), 0, s, R, K, d, scores, W, b, Y, xs);
    }
    return check_launch("score_embed", (double)R * (8.0 * K + 4.0 * d + 4.0 * K), 2.0 * R * K * d);
}

// Backward of score_embeddings: gW[c,k] += sum_r dY[r,c] xs[r,k],  gb[c] += sum_r dY[r,c].  One pass over dY (the
// product has only K <= 8 columns, so a warp keeps its share of gW in registers: lane = output channel), summed per CTA
// in shared memory, one global atomic per entry and CTA (the 9 x d addresses sit in a handful of L2 lines, so the number
// of CTAs, not the bytes, sets the cost of that tail).
constexpr int SEB_K = 8;
constexpr int SEB_THREADS = 768;               // one CTA per SM: the atomics at the end are per CTA, so few large CTAs
template <bool WIDE>                           // WIDE: d > 32, a second channel per lane
__global__ void __launch_bounds__(SEB_THREADS, 1) score_embed_bwd_kernel(int64_t R, int K, int d, const float* __restrict__ dY,
                                                                          int64_t lddy, const float* __restrict__ xs,
                                                                          float* gW, float* gb) {
    __shared__ float red[SEB_K + 1][64];
    for (int e = threadIdx.x; e < (SEB_K + 1) * 64; e += blockDim.x) (&red[0][0])[e] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float a0[SEB_K + 1], a1[SEB_K + 1];        // [k] = weight gradient column k, [SEB_K] = bias gradient
#pragma unroll
    for (int k = 0; k <= SEB_K; ++k) a0[k] = a1[k] = 0.f;
    const bool c0 = lane < d, c1 = WIDE && lane + 32 < d;
    constexpr int U = 8;                       // rows in flight per warp (the loop is otherwise one 128-byte load deep)
    for (int64_t rb = warp * U; rb < R; rb += nwarps * U) {
        float g0[U], g1[U], xv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t r = rb + u;
            const bool live = r < R;
            g0[u] = (live && c0) ? dY[r * lddy + lane] : 0.f;
            g1[u] = (WIDE && live && c1) ? dY[r * lddy + lane + 32] : 0.f;
            xv[u] = (live && lane < K) ? xs[r * K + lane] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int k = 0; k < SEB_K; ++k) {
                const float x = __shfl_sync(0xffffffffu, xv[u], k);
                a0[k] = fmaf(g0[u], x, a0[k]);
                if (WIDE) a1[k] = fmaf(g1[u], x, a1[k]);
            }
            a0[SEB_K] += g0[u];
            if (WIDE) a1[SEB_K] += g1[u];
        }
    }
#pragma unroll
    for (int k = 0; k <= SEB_K; ++k) {
        if (k < SEB_K && k >= K) continue;
        if (c0) atomicAdd(&red[k][lane], a0[k]);
        if (c1) atomicAdd(&red[k][lane + 32], a1[k]);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < (SEB_K + 1) * 64; e += blockDim.x) {
        const int k = e >> 6, c = e & 63;
        if (c >= d || (k < SEB_K && k >= K)) continue;
        const float t = red[k][c];
        if (t == 0.f) continue;
        if (k < SEB_K) atomicAdd(gW + (int64_t)c * K + k, t);
        else if (gb) atomicAdd(gb + c, t);
    }
}

bool score_embed_bwd_ok(int K, int d) { return K <= SEB_K && d <= 64; }

int score_embed_bwd(int64_t R, int K, int d, const float* dY, int64_t lddy, const float* xs, float* gW, float* gb,
                    cudaStream_t s) {
    if (R <= 0) return INTEL_OK;
    INTEL_REQUIRE(score_embed_bwd_ok(K, d), INTEL_ERR_UNSUPPORTED, "score_embed_bwd: model_num %d / s_emb_size %d", K, d);
    unsigned grid = stream_grid(ceil_div(R, (SEB_THREADS / 32) * 8), 1);
    if (d > 32) {
        LAUNCH(score_embed_bwd_kernel<true>, dim3(grid), dim3(SEB_THREADS), 0, s, R, K, d, dY, lddy, xs, gW, gb);
    } else {
        LAUNCH(score_embed_bwd_kernel<false>, dim3(grid), dim3(SEB_THREADS), 0, s, R, K, d, dY, lddy, xs, gW, gb);
    }
    return check_launch("score_embed_bwd", (double)R * (4.0 * d + 4.0 * K), 2.0 * R * K * d);
}

// ------------------------------------------------------------------------------------------------
// BERT4RecEncoder learned positions (GeneralSeq.py:93-96): position index is t for live slots, 0 for pads
__global__ void __launch_bounds__(256) add_pos_kernel(int64_t B, int64_t T, int d, const int64_t* __restrict__ lens,
                                                      const float* __restrict__ pos, float* seq) {
    const int64_t total = B * T * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % d);
        const int64_t bt = e / d;
        const int64_t t = bt % T, bb = bt / T;
        const int64_t p = (t < lens[bb]) ? t : 0;
        seq[e] += pos[p * d + c];
    }
}
int add_positions(int64_t B, int64_t T, int d, const int64_t* lens, const float* pos, float* seq, cudaStream_t s) {
    if (B * T <= 0) return INTEL_OK;
    unsigned grid = stream_grid(ceil_div(B * T * d, 256), 8);
    LAUNCH(add_pos_kernel, dim3(grid), dim3(256), 0, s, B, T, d, lens, pos, seq);
    return check_launch("add_positions");
}

__global__ void __launch_bounds__(256) add_pos_bwd_kernel(int64_t B, int64_t T, int d, const int64_t* __restrict__ lens,
                                                          const float* __restrict__ d_seq, float* d_pos) {
    const int64_t total = B * T * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % d);
        const int64_t bt = e / d;
        const int64_t t = bt % T, bb = bt / T;
        const int64_t p = (t < lens[bb]) ? t : 0;
        const float g = d_seq[e];
        if (g != 0.f) atomicAdd(d_pos + p * d + c, g);
    }
}
int add_positions_bwd(int64_t B, int64_t T, int d, const int64_t* lens, const float* d_seq, float* d_pos,
                      cudaStream_t s) {
    if (B * T <= 0) return INTEL_OK;
    unsigned grid = stream_grid(ceil_div(B * T * d, 256), 8);
    LAUNCH(add_pos_bwd_kernel, dim3(grid), dim3(256), 0, s, B, T, d, lens, d_seq, d_pos);
    return check_launch("add_positions_bwd");
}

// his_vector = seq[b, len-1]  (GeneralSeq.py:105)
__global__ void __launch_bounds__(256) take_last_kernel(int64_t B, int64_t T, int d, const int64_t* __restrict__ lens,
                                                        const float* __restrict__ X, float* out, int64_t ld_out, int bwd) {
    const int64_t total = B * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % d);
        const int64_t bb = e / d;
        int64_t t = lens[bb] - 1;
        if (t < 0) t = 0;
        if (t >= T) t = T - 1;
        if (!bwd) out[bb * ld_out + c] = X[(bb * T + t) * d + c];
        else const_cast<float*>(X)[(bb * T + t) * d + c] = out[bb * ld_out + c];
    }
}
int take_last(int64_t B, int64_t T, int d, const int64_t* lens, const float* X, float* out, int64_t ld_out,
              cudaStream_t s) {
    if (B <= 0) return INTEL_OK;
    unsigned grid = stream_grid(ceil_div(B * d, 256), 8);
    LAUNCH(take_last_kernel, dim3(grid), dim3(256), 0, s, B, T, d, lens, X, out, ld_out, 0);
    return check_launch("take_last");
}
int take_last_bwd(int64_t B, int64_t T, int d, const int64_t* lens, const float* d_out, int64_t ld, float* dX,
                  cudaStream_t s) {
    if (B <= 0) return INTEL_OK;
    unsigned grid = stream_grid(ceil_div(B * d, 256), 8);
    LAUNCH(take_last_kernel, dim3(grid), dim3(256), 0, s, B, T, d, lens, (const float*)dX, const_cast<float*>(d_out), ld, 1);
    return check_launch("take_last_bwd");
}

int copy_d2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (!bytes) return INTEL_OK;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) { set_error("cudaMemcpyAsync: %s", cudaGetErrorString(e)); return INTEL_ERR_CUDA; }
    return INTEL_OK;
}

int fill_zero(void* p, size_t bytes, cudaStream_t s) {
    if (!bytes) return INTEL_OK;
    cudaError_t e = cudaMemsetAsync(p, 0, bytes, s);
    if (e != cudaSuccess) { set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return INTEL_ERR_CUDA; }
    return INTEL_OK;
}

}  // namespace intel
