// Optimizer step of the training loop (BaseRunner._build_optimizer, BaseRunner.py:182-188: torch.optim.Adam over
// BaseModel.customize_parameters' two groups, BaseModel.py:53-62 - L2 on the weights, none on the biases).
// One launch updates up to ADAM_MAX_TENSORS parameter tensors (torch's unfused Adam issues ~10 small kernels per
// tensor).  The arithmetic follows torch.optim.Adam's single-tensor path operation by operation (separately
// rounded multiplies and adds, lerp for the first moment); torch's own kernels may contract some of them into
// FMAs, so parity is to the last ulp or two, not bitwise.
#include "kernels.h"
#include "../../include/intel_b200.h"

namespace intel {

static const int ADAM_MAX_TENSORS = 48;

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
    float lr_over_bc1;      // lr / (1 - beta1^step)
    float bc2_sqrt;         // sqrt(1 - beta2^step)
    float beta2, eps;
    float w1, w2;           // 1 - beta1, 1 - beta2, rounded from double like torch's python-side scalars
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
    const float w1 = a.w1, w2 = a.w2, ns = -a.lr_over_bc1;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    const bool vec = ((((uintptr_t)t.p) | ((uintptr_t)t.g) | ((uintptr_t)t.m) | ((uintptr_t)t.v)) & 15) == 0;
    const int64_t n4 = vec ? t.n / 4 : 0;
    for (int64_t i = tid; i < n4; i += nth) {           // 16-byte accesses: 7 streams of 4 floats per thread in flight
        float4 p = reinterpret_cast<float4*>(t.p)[i], m = reinterpret_cast<float4*>(t.m)[i], v = reinterpret_cast<float4*>(t.v)[i];
        const float4 g = reinterpret_cast<const float4*>(t.g)[i];
        adam_one(p.x, g.x, m.x, v.x, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
        adam_one(p.y, g.y, m.y, v.y, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
        adam_one(p.z, g.z, m.z, v.z, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
        adam_one(p.w, g.w, m.w, v.w, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
        reinterpret_cast<float4*>(t.p)[i] = p;
        reinterpret_cast<float4*>(t.m)[i] = m;
        reinterpret_cast<float4*>(t.v)[i] = v;
    }
    for (int64_t i = 4 * n4 + tid; i < t.n; i += nth) {
        float p = t.p[i], m = t.m[i], v = t.v[i];
        adam_one(p, t.g[i], m, v, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
        t.p[i] = p;
        t.m[i] = m;
        t.v[i] = v;
    }
}

// Row-wise step of a sparse (row set) gradient: rows[r] of p / m / v get adam_one with the compact gradient row r; every
// other row keeps p, m and v bit for bit.  The arithmetic per element is the dense kernel's, so a row updated here equals
// the same row updated by adam_kernel with that gradient.
struct AdamRowsTensor {
    float* p;
    const float* g;        // [U, d]
    float* m;
    float* v;
    const int64_t* rows;   // [U], distinct
    int64_t U;
    int d;
    float wd;
};
struct AdamRowsArgs {
    AdamRowsTensor t[ADAM_MAX_TENSORS];
    int count;
    float lr_over_bc1, bc2_sqrt, beta2, eps, w1, w2;
};

__global__ void __launch_bounds__(256) adam_rows_kernel(AdamRowsArgs a) {
    const AdamRowsTensor t = a.t[blockIdx.y];
    const float w1 = a.w1, w2 = a.w2, ns = -a.lr_over_bc1;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    const bool vec = t.d % 4 == 0 && ((((uintptr_t)t.p) | ((uintptr_t)t.g) | ((uintptr_t)t.m) | ((uintptr_t)t.v)) & 15) == 0;
    if (vec) {
        const int per_row = t.d / 4;
        for (int64_t e = tid; e < t.U * per_row; e += nth) {
            const int64_t r = e / per_row, row = t.rows[r];
            const int c = (int)(e % per_row);
            float4* pp = reinterpret_cast<float4*>(t.p + row * t.d) + c;
            float4* mp = reinterpret_cast<float4*>(t.m + row * t.d) + c;
            float4* vp = reinterpret_cast<float4*>(t.v + row * t.d) + c;
            float4 p = *pp, m = *mp, v = *vp;
            const float4 g = reinterpret_cast<const float4*>(t.g + r * t.d)[c];
            adam_one(p.x, g.x, m.x, v.x, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
            adam_one(p.y, g.y, m.y, v.y, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
            adam_one(p.z, g.z, m.z, v.z, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
            adam_one(p.w, g.w, m.w, v.w, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
            *pp = p;
            *mp = m;
            *vp = v;
        }
    } else {
        for (int64_t e = tid; e < t.U * t.d; e += nth) {
            const int64_t r = e / t.d, i = t.rows[r] * t.d + e % t.d;
            float p = t.p[i], m = t.m[i], v = t.v[i];
            adam_one(p, t.g[e], m, v, t.wd, w1, w2, a.beta2, a.bc2_sqrt, a.eps, ns);
            t.p[i] = p;
            t.m[i] = m;
            t.v[i] = v;
        }
    }
}

int adam_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq, const int64_t* const* rows,
                   const float* const* grads, const int64_t* nrows, const int32_t* dim, const float* weight_decay, double lr,
                   double beta1_d, double beta2_d, double eps_d, int64_t step, cudaStream_t s) {
    INTEL_REQUIRE(count >= 0 && step >= 1, INTEL_ERR_ARG, "adam_rows_step: bad count / step");
    const double bc1 = 1.0 - pow(beta1_d, (double)step), bc2 = 1.0 - pow(beta2_d, (double)step);
    AdamRowsArgs a;
    memset(&a, 0, sizeof(a));
    a.lr_over_bc1 = (float)(lr / bc1);             // the scalars exactly as adam_step forms them
    a.bc2_sqrt = (float)sqrt(bc2);
    a.beta2 = (float)beta2_d; a.eps = (float)eps_d;
    a.w1 = (float)(1.0 - (double)beta1_d);
    a.w2 = (float)(1.0 - (double)beta2_d);
    int64_t widest = 1;
    auto flush = [&]() -> int {
        if (a.count == 0) return INTEL_OK;
        int64_t bx = ceil_div(widest, 256 * 4);
        if (bx > 16 * kNumSMs) bx = 16 * kNumSMs;
        LAUNCH(adam_rows_kernel, dim3((unsigned)bx, (unsigned)a.count), dim3(256), 0, s, a);
        double bytes = 0;
        for (int i = 0; i < a.count; ++i) bytes += (double)a.t[i].U * (28.0 * a.t[i].d + 8.0);
        a.count = 0;
        widest = 1;
        return check_launch("adam_rows", bytes, 0.0);
    };
    for (int i = 0; i < count; ++i) {
        INTEL_REQUIRE(nrows[i] >= 0 && dim[i] > 0 && (nrows[i] == 0 || (params[i] && exp_avg[i] && exp_avg_sq[i] && rows[i] && grads[i])),
                      INTEL_ERR_ARG, "adam_rows_step: bad tensor %d", i);
        if (nrows[i] == 0) continue;
        a.t[a.count++] = AdamRowsTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], rows[i], nrows[i], dim[i], weight_decay[i]};
        if (nrows[i] * dim[i] > widest) widest = nrows[i] * dim[i];
        if (a.count == ADAM_MAX_TENSORS) INTEL_TRY(flush());
    }
    return flush();
}

int adam_step(int count, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
              const int64_t* numel, const float* weight_decay, double lr, double beta1_d, double beta2_d, double eps_d, int64_t step,
              cudaStream_t s) {
    const float beta2 = (float)beta2_d, eps = (float)eps_d;
    INTEL_REQUIRE(count >= 0 && step >= 1, INTEL_ERR_ARG, "adam_step: bad count / step");
    const double bc1 = 1.0 - pow(beta1_d, (double)step), bc2 = 1.0 - pow(beta2_d, (double)step);
    AdamArgs a;
    memset(&a, 0, sizeof(a));
    a.lr_over_bc1 = (float)(lr / bc1);
    a.bc2_sqrt = (float)sqrt(bc2);
    a.beta2 = beta2; a.eps = eps;
    a.w1 = (float)(1.0 - (double)beta1_d);
    a.w2 = (float)(1.0 - (double)beta2_d);
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
