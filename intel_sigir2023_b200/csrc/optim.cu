// Optimizer step of the training loop (BaseRunner._build_optimizer, BaseRunner.py:182-188: torch.optim.Adam over
// BaseModel.customize_parameters' two groups, BaseModel.py:53-62 - L2 on the weights, none on the biases).
// One launch updates up to ADAM_MAX_TENSORS parameter tensors (torch's unfused Adam issues ~10 small kernels per
// tensor).  The arithmetic follows torch.optim.Adam's single-tensor path operation by operation (separately
// rounded multiplies and adds, lerp for the first moment); torch's own kernels may contract some of them into
// FMAs, so parity is to the last ulp or two, not bitwise.
#include <vector>

#include "kernels.h"
#include "../../include/intel_b200.h"

namespace intel {

static const int ADAM_MAX_TENSORS = 48;

// The float32 scalars of one Adam step.  Every step forms them with adam_scalars only: the deferred row-wise step is
// bitwise the dense one because its replayed updates use exactly the floats the dense step would have used.
struct AdamScalars {
    float lr_over_bc1;      // lr / (1 - beta1^step)
    float bc2_sqrt;         // sqrt(1 - beta2^step)
    float beta2, eps;
    float w1, w2;           // 1 - beta1, 1 - beta2
};

// computed in double and rounded once, like torch's python-side scalars
static AdamScalars adam_scalars(double lr, double beta1, double beta2, double eps, int64_t step) {
    const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
    return AdamScalars{(float)(lr / bc1), (float)sqrt(bc2), (float)beta2, (float)eps, (float)(1.0 - beta1), (float)(1.0 - beta2)};
}

struct AdamTensor {
    float* p;
    const float* g;
    float* m;
    float* v;
    int64_t n;
    float wd;
};
struct AdamArgs {
    AdamTensor t[ADAM_MAX_TENSORS];
    int count;
    AdamScalars s;
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float wd, float w1, float w2, float beta2,
                                         float bc2_sqrt, float eps, float neg_step) {
    if (wd != 0.f) g = __fadd_rn(g, __fmul_rn(p, wd));                       // grad.add(param, alpha=weight_decay)
    m = __fadd_rn(m, __fmul_rn(w1, __fadd_rn(g, -m)));                       // exp_avg.lerp_(grad, 1 - beta1)
    v = __fadd_rn(__fmul_rn(v, beta2), __fmul_rn(__fmul_rn(w2, g), g));      // mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), eps);
    p = __fadd_rn(p, __fmul_rn(neg_step, __fdiv_rn(m, denom)));              // addcdiv_(exp_avg, denom, value=-step_size)
}

__global__ void __launch_bounds__(256) adam_kernel(AdamArgs a) {
    const AdamTensor t = a.t[blockIdx.y];
    const AdamScalars& s = a.s;
    const float w1 = s.w1, w2 = s.w2, ns = -s.lr_over_bc1;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    const bool vec = ((((uintptr_t)t.p) | ((uintptr_t)t.g) | ((uintptr_t)t.m) | ((uintptr_t)t.v)) & 15) == 0;
    const int64_t n4 = vec ? t.n / 4 : 0;
    for (int64_t i = tid; i < n4; i += nth) {           // 16-byte accesses: 7 streams of 4 floats per thread in flight
        float4 p = reinterpret_cast<float4*>(t.p)[i], m = reinterpret_cast<float4*>(t.m)[i], v = reinterpret_cast<float4*>(t.v)[i];
        const float4 g = reinterpret_cast<const float4*>(t.g)[i];
        adam_one(p.x, g.x, m.x, v.x, t.wd, w1, w2, s.beta2, s.bc2_sqrt, s.eps, ns);
        adam_one(p.y, g.y, m.y, v.y, t.wd, w1, w2, s.beta2, s.bc2_sqrt, s.eps, ns);
        adam_one(p.z, g.z, m.z, v.z, t.wd, w1, w2, s.beta2, s.bc2_sqrt, s.eps, ns);
        adam_one(p.w, g.w, m.w, v.w, t.wd, w1, w2, s.beta2, s.bc2_sqrt, s.eps, ns);
        reinterpret_cast<float4*>(t.p)[i] = p;
        reinterpret_cast<float4*>(t.m)[i] = m;
        reinterpret_cast<float4*>(t.v)[i] = v;
    }
    for (int64_t i = 4 * n4 + tid; i < t.n; i += nth) {
        float p = t.p[i], m = t.m[i], v = t.v[i];
        adam_one(p, t.g[i], m, v, t.wd, w1, w2, s.beta2, s.bc2_sqrt, s.eps, ns);
        t.p[i] = p;
        t.m[i] = m;
        t.v[i] = v;
    }
}

// Row-wise steps of a sparse (row set) gradient, one kernel in four modes.  The listed rows of p / m / v get adam_one per
// element, the dense kernel's arithmetic; every other row keeps p, m and v bit for bit.
// LAZY:     listed rows take the update with their compact gradient row (done / hist unused), so a row updated here
//           equals the same row updated by adam_kernel with that gradient.
// The other three modes are the deferred (exact) step.  Dense Adam gives every row a step never names a gradient of
// exactly +0.0, and such an update depends only on the row's own p / m / v and that step's scalars.  So the updates a row
// skips are deferred and replayed later, in order, through the same adam_one: a row with k pending updates is read and
// written once, and the result is bitwise the dense one.  Per tensor the caller keeps
//   hist [>= n, 8] float: entry k holds the scalars of update k + 1 (ADAM_HIST_* below),
//   done [rows] int32:    how many of the n updates row r has received (the row is current when done[r] == n).
// STEP:     listed rows replay done[r] .. n-2 with g = +0.0, then take update n with their gradient row; the kernel also
//           stores update n's scalars (its arguments) to hist[n-1].
// CATCH_UP: listed rows (the count read from device memory) replay done[r] .. n-1.
// FLUSH:    every row replays done[r] .. n-1, and done is reset to 0 for the caller to restart its count.
// A row is handled by one group of G lanes of a warp (G = the power of two >= the row's vectors, at most 32).  In the
// deferred modes its lanes read done[r] before the group's first lane writes it, with a __syncwarp in between, so the
// loop is warp-uniform.
enum { ADAM_HIST_LR_BC1, ADAM_HIST_BC2_SQRT, ADAM_HIST_BETA2, ADAM_HIST_EPS, ADAM_HIST_W1, ADAM_HIST_W2, ADAM_HIST_WD, ADAM_HIST_WIDTH = 8 };
enum AdamRowsMode { ADAM_ROWS_LAZY, ADAM_DEFERRED_STEP, ADAM_DEFERRED_CATCH_UP, ADAM_DEFERRED_FLUSH };

// the modes that apply a new update with a gradient row
__host__ __device__ constexpr bool adam_rows_take_grad(int mode) { return mode == ADAM_ROWS_LAZY || mode == ADAM_DEFERRED_STEP; }

struct AdamDeferredTensor {
    float* p;
    const float* g;          // [U, d] (LAZY, STEP)
    float* m;
    float* v;
    const int64_t* rows;     // [U] distinct; NULL: rows 0 .. U-1 (FLUSH)
    const int64_t* count;    // CATCH_UP: device count of rows (<= U)
    int32_t* done;           // NULL in LAZY
    float* hist;             // NULL in LAZY
    int64_t U;
    int d;
    int n;
    float wd;
};
struct AdamDeferredArgs {
    AdamDeferredTensor t[ADAM_MAX_TENSORS];
    int count;
    AdamScalars s;           // LAZY, STEP: the scalars of the new update
};

// V consecutive elements of one row: replay hist[k0 .. k1) with g = +0.0 (REPLAY), then one update with the gradient g_ (GRAD)
template <bool REPLAY, bool GRAD, int V>
__device__ __forceinline__ void adam_rows_elems(float* p_, float* m_, float* v_, const float* g_, const float* hist, int k0, int k1,
                                                float wd, const AdamScalars& s) {
    float p[V], m[V], v[V];
    if constexpr (V == 4) {
        const float4 P = *reinterpret_cast<const float4*>(p_), M = *reinterpret_cast<const float4*>(m_),
                     W = *reinterpret_cast<const float4*>(v_);
        p[0] = P.x; p[1] = P.y; p[2] = P.z; p[3] = P.w;
        m[0] = M.x; m[1] = M.y; m[2] = M.z; m[3] = M.w;
        v[0] = W.x; v[1] = W.y; v[2] = W.z; v[3] = W.w;
    } else {
        p[0] = *p_; m[0] = *m_; v[0] = *v_;
    }
    if constexpr (REPLAY) {
        for (int k = k0; k < k1; ++k) {
            const float4 h0 = reinterpret_cast<const float4*>(hist)[2 * k], h1 = reinterpret_cast<const float4*>(hist)[2 * k + 1];
#pragma unroll
            for (int j = 0; j < V; ++j) adam_one(p[j], 0.0f, m[j], v[j], h1.z, h1.x, h1.y, h0.z, h0.y, h0.w, -h0.x);
        }
    }
    if constexpr (GRAD) {
        float g[V];
        if constexpr (V == 4) {
            const float4 G = *reinterpret_cast<const float4*>(g_);
            g[0] = G.x; g[1] = G.y; g[2] = G.z; g[3] = G.w;
        } else {
            g[0] = *g_;
        }
#pragma unroll
        for (int j = 0; j < V; ++j) adam_one(p[j], g[j], m[j], v[j], wd, s.w1, s.w2, s.beta2, s.bc2_sqrt, s.eps, -s.lr_over_bc1);
    }
    if constexpr (V == 4) {
        *reinterpret_cast<float4*>(p_) = make_float4(p[0], p[1], p[2], p[3]);
        *reinterpret_cast<float4*>(m_) = make_float4(m[0], m[1], m[2], m[3]);
        *reinterpret_cast<float4*>(v_) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        *p_ = p[0]; *m_ = m[0]; *v_ = v[0];
    }
}

template <int MODE, int V>
__device__ __forceinline__ void adam_rows_groups(const AdamDeferredTensor& t, const AdamScalars& s, int64_t U) {
    constexpr bool LAZY = MODE == ADAM_ROWS_LAZY, GRAD = adam_rows_take_grad(MODE);
    const int per_row = t.d / V;
    int G = 1;
    while (G < per_row && G < 32) G <<= 1;
    const int lane = threadIdx.x & 31, lg = lane & (G - 1), rows_per_warp = 32 / G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int last = MODE == ADAM_DEFERRED_STEP ? t.n - 1 : t.n;        // replay hist[done .. last)
    for (int64_t base = warp * rows_per_warp; base < U; base += nwarps * rows_per_warp) {
        const int64_t r = base + lane / G;
        const bool live = r < U;
        int64_t row = 0;
        int k0 = last;
        if (live) {
            row = t.rows != nullptr ? t.rows[r] : r;
            if constexpr (!LAZY) k0 = t.done[row];
        }
        if (live && (GRAD || k0 < last)) {
            for (int c = lg; c < per_row; c += G) {
                const int64_t e = row * t.d + (int64_t)c * V;
                adam_rows_elems<!LAZY, GRAD, V>(t.p + e, t.m + e, t.v + e, GRAD ? t.g + r * t.d + (int64_t)c * V : nullptr, t.hist, k0,
                                                last, t.wd, s);
            }
        }
        if constexpr (!LAZY) {
            __syncwarp();
            if (live && lg == 0) {
                if (MODE == ADAM_DEFERRED_FLUSH) t.done[row] = 0;
                else if (MODE == ADAM_DEFERRED_STEP || k0 < last) t.done[row] = t.n;
            }
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(256) adam_rows_kernel(AdamDeferredArgs a) {
    const AdamDeferredTensor t = a.t[blockIdx.y];
    int64_t U = t.U;
    if (MODE == ADAM_DEFERRED_CATCH_UP) U = min(U, *t.count);
    if (MODE == ADAM_DEFERRED_STEP && blockIdx.x == 0 && threadIdx.x == 0) {
        float* h = t.hist + (int64_t)(t.n - 1) * ADAM_HIST_WIDTH;     // no lane of this launch reads entry n-1
        h[ADAM_HIST_LR_BC1] = a.s.lr_over_bc1; h[ADAM_HIST_BC2_SQRT] = a.s.bc2_sqrt; h[ADAM_HIST_BETA2] = a.s.beta2;
        h[ADAM_HIST_EPS] = a.s.eps; h[ADAM_HIST_W1] = a.s.w1; h[ADAM_HIST_W2] = a.s.w2; h[ADAM_HIST_WD] = t.wd; h[7] = 0.f;
    }
    const bool vec = t.d % 4 == 0 && ((((uintptr_t)t.p) | ((uintptr_t)t.m) | ((uintptr_t)t.v) |
                                       (adam_rows_take_grad(MODE) ? (uintptr_t)t.g : 0)) & 15) == 0;
    if (vec) adam_rows_groups<MODE, 4>(t, a.s, U);
    else adam_rows_groups<MODE, 1>(t, a.s, U);
}

// one launch per ADAM_MAX_TENSORS tensors, grid sized for the widest (rows x d).  STEP keeps tensors without rows: their
// launch still records the update's scalars.
template <int MODE>
static int adam_rows_launch(const AdamScalars& sc, const std::vector<AdamDeferredTensor>& ts, cudaStream_t s, const char* name) {
    const double elem_bytes = adam_rows_take_grad(MODE) ? 28.0 : 24.0, row_bytes = MODE == ADAM_ROWS_LAZY ? 8.0 : 16.0;
    AdamDeferredArgs a;
    memset(&a, 0, sizeof(a));
    a.s = sc;
    int64_t widest = 1;
    double bytes = 0;
    for (size_t i = 0; i < ts.size(); ++i) {
        a.t[a.count++] = ts[i];
        if (ts[i].U * ts[i].d > widest) widest = ts[i].U * ts[i].d;
        bytes += (double)ts[i].U * (elem_bytes * ts[i].d + row_bytes);
        if (a.count < ADAM_MAX_TENSORS && i + 1 < ts.size()) continue;
        int64_t bx = ceil_div(widest, 256 * 4);
        if (bx > 16 * kNumSMs) bx = 16 * kNumSMs;
        LAUNCH(adam_rows_kernel<MODE>, dim3((unsigned)bx, (unsigned)a.count), dim3(256), 0, s, a);
        INTEL_TRY(check_launch(name, bytes, 0.0));
        a.count = 0;
        widest = 1;
        bytes = 0;
    }
    return INTEL_OK;
}

int adam_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq, const int64_t* const* rows,
                   const float* const* grads, const int64_t* nrows, const int32_t* dim, const float* weight_decay, double lr,
                   double beta1_d, double beta2_d, double eps_d, int64_t step, cudaStream_t s) {
    INTEL_REQUIRE(count >= 0 && step >= 1, INTEL_ERR_ARG, "adam_rows_step: bad count / step");
    std::vector<AdamDeferredTensor> ts;
    for (int i = 0; i < count; ++i) {
        INTEL_REQUIRE(nrows[i] >= 0 && dim[i] > 0 && (nrows[i] == 0 || (params[i] && exp_avg[i] && exp_avg_sq[i] && rows[i] && grads[i])),
                      INTEL_ERR_ARG, "adam_rows_step: bad tensor %d", i);
        if (nrows[i] == 0) continue;
        ts.push_back(AdamDeferredTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], rows[i], nullptr, nullptr, nullptr, nrows[i],
                                        dim[i], 0, weight_decay[i]});
    }
    return adam_rows_launch<ADAM_ROWS_LAZY>(adam_scalars(lr, beta1_d, beta2_d, eps_d, step), ts, s, "adam_rows");
}

int adam_deferred_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                            const int64_t* const* rows, const float* const* grads, const int64_t* nrows, const int32_t* dim,
                            const float* weight_decay, int32_t* const* done, float* const* hist, const int32_t* n_updates,
                            double lr, double beta1_d, double beta2_d, double eps_d, int64_t step, cudaStream_t s) {
    INTEL_REQUIRE(count >= 0 && step >= 1, INTEL_ERR_ARG, "adam_deferred_rows_step: bad count / step");
    std::vector<AdamDeferredTensor> ts;
    for (int i = 0; i < count; ++i) {
        INTEL_REQUIRE(nrows[i] >= 0 && dim[i] > 0 && n_updates[i] >= 1 && params[i] && exp_avg[i] && exp_avg_sq[i] && done[i] &&
                      hist[i] && (nrows[i] == 0 || (rows[i] && grads[i])),
                      INTEL_ERR_ARG, "adam_deferred_rows_step: bad tensor %d", i);
        ts.push_back(AdamDeferredTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], rows[i], nullptr, done[i], hist[i], nrows[i],
                                        dim[i], n_updates[i], weight_decay[i]});
    }
    return adam_rows_launch<ADAM_DEFERRED_STEP>(adam_scalars(lr, beta1_d, beta2_d, eps_d, step), ts, s, "adam_deferred_step");
}

int adam_deferred_catch_up(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                           const int64_t* const* rows, const int64_t* const* row_count, const int64_t* nrows, const int32_t* dim,
                           int32_t* const* done, const float* const* hist, const int32_t* n_updates, cudaStream_t s) {
    INTEL_REQUIRE(count >= 0, INTEL_ERR_ARG, "adam_deferred_catch_up: bad count");
    std::vector<AdamDeferredTensor> listed, all;
    for (int i = 0; i < count; ++i) {
        INTEL_REQUIRE(nrows[i] >= 0 && dim[i] > 0 && n_updates[i] >= 0, INTEL_ERR_ARG, "adam_deferred_catch_up: bad tensor %d", i);
        if (nrows[i] == 0 || n_updates[i] == 0) continue;              // nothing is pending
        INTEL_REQUIRE(params[i] && exp_avg[i] && exp_avg_sq[i] && done[i] && hist[i] && (rows[i] == nullptr || row_count[i]),
                      INTEL_ERR_ARG, "adam_deferred_catch_up: null pointer in tensor %d", i);
        (rows[i] ? listed : all).push_back(AdamDeferredTensor{params[i], nullptr, exp_avg[i], exp_avg_sq[i], rows[i], row_count[i],
                                                              done[i], const_cast<float*>(hist[i]), nrows[i], dim[i], n_updates[i],
                                                              0.f});
    }
    INTEL_TRY(adam_rows_launch<ADAM_DEFERRED_CATCH_UP>(AdamScalars{}, listed, s, "adam_deferred_catch_up"));
    return adam_rows_launch<ADAM_DEFERRED_FLUSH>(AdamScalars{}, all, s, "adam_deferred_flush");
}

int adam_step(int count, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
              const int64_t* numel, const float* weight_decay, double lr, double beta1_d, double beta2_d, double eps_d, int64_t step,
              cudaStream_t s) {
    INTEL_REQUIRE(count >= 0 && step >= 1, INTEL_ERR_ARG, "adam_step: bad count / step");
    AdamArgs a;
    memset(&a, 0, sizeof(a));
    a.s = adam_scalars(lr, beta1_d, beta2_d, eps_d, step);
    // big tensors (embedding tables) get a launch of their own with a full grid; all small tensors share launches of
    // up to ADAM_MAX_TENSORS tensors with a short grid (a common grid sized for the largest tensor would schedule tens of
    // thousands of empty blocks)
    const int64_t big = (int64_t)1 << 18;
    auto flush = [&](int64_t widest) -> int {
        if (a.count == 0) return INTEL_OK;
        int64_t bx = ceil_div(widest, 256 * 4);
        if (bx > 16 * kNumSMs) bx = 16 * kNumSMs;
        LAUNCH(adam_kernel, dim3((unsigned)bx, (unsigned)a.count), dim3(256), 0, s, a);
        double bytes = 0;
        for (int i = 0; i < a.count; ++i) bytes += 28.0 * (double)a.t[i].n;
        a.count = 0;
        return check_launch("adam", bytes, 0.0);
    };
    for (int i = 0; i < count; ++i) {
        if (numel[i] < big) continue;
        a.t[0] = AdamTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], numel[i], weight_decay[i]};
        a.count = 1;
        INTEL_TRY(flush(numel[i]));
    }
    int64_t widest = 1;
    for (int i = 0; i < count; ++i) {
        if (numel[i] >= big || numel[i] <= 0) continue;
        a.t[a.count++] = AdamTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], numel[i], weight_decay[i]};
        if (numel[i] > widest) widest = numel[i];
        if (a.count == ADAM_MAX_TENSORS) { INTEL_TRY(flush(widest)); widest = 1; }
    }
    INTEL_TRY(flush(widest));
    return INTEL_OK;
}

}  // namespace intel

using namespace intel;

int intel_adam_step(int count, float* const* params, const float* const* grads, float* const* exp_avg,
                    float* const* exp_avg_sq, const int64_t* numel, const float* weight_decay, double lr, double beta1,
                    double beta2, double eps, int64_t step, intel_stream_t stream) {
    return adam_step(count, params, grads, exp_avg, exp_avg_sq, numel, weight_decay, lr, beta1, beta2, eps, step, (cudaStream_t)stream);
}

int intel_adam_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                         const int64_t* const* rows, const float* const* grads, const int64_t* nrows, const int32_t* dim,
                         const float* weight_decay, double lr, double beta1, double beta2, double eps, int64_t step,
                         intel_stream_t stream) {
    return adam_rows_step(count, params, exp_avg, exp_avg_sq, rows, grads, nrows, dim, weight_decay, lr, beta1, beta2, eps, step,
                          (cudaStream_t)stream);
}

int intel_adam_deferred_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                                  const int64_t* const* rows, const float* const* grads, const int64_t* nrows, const int32_t* dim,
                                  const float* weight_decay, int32_t* const* done, float* const* hist, const int32_t* n_updates,
                                  double lr, double beta1, double beta2, double eps, int64_t step, intel_stream_t stream) {
    return adam_deferred_rows_step(count, params, exp_avg, exp_avg_sq, rows, grads, nrows, dim, weight_decay, done, hist, n_updates,
                                   lr, beta1, beta2, eps, step, (cudaStream_t)stream);
}

int intel_adam_deferred_catch_up(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                                 const int64_t* const* rows, const int64_t* const* row_count, const int64_t* nrows,
                                 const int32_t* dim, int32_t* const* done, const float* const* hist, const int32_t* n_updates,
                                 intel_stream_t stream) {
    return adam_deferred_catch_up(count, params, exp_avg, exp_avg_sq, rows, row_count, nrows, dim, done, hist, n_updates,
                                  (cudaStream_t)stream);
}
