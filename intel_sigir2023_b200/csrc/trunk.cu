// Fused self-attention stack of IntEL.predict_ensemble (IntEL.py:182-197, layers.py:31-60) for the shape
// every script of the reference uses: stream width d = 32, list length L <= 64.
//
// A session's whole N-layer stack runs inside one kernel.  A warp owns 16 tokens and keeps their activations
// in the accumulator layout of the m16n8k8 TF32 MMA; every product is a 3xTF32 tensor-core MMA (mma.cuh) and the
// output tile of one product is re-used as the A operand of the next without leaving registers.  Shared memory
// holds the weights and what the warps of a session must exchange (K / V rows; in the backward pass also the
// tiles that are contracted over tokens).  The forward pass saves q|k|v, the attention output, the FFN hidden,
// the pre-LN sum and the LN statistics of each layer for the backward pass, which replays only the softmax.
// Weight gradients stay in registers across all sessions of a CTA and are flushed once per CTA.
#include "kernels.h"
#include "mma.cuh"
#include "tc05.cuh"

namespace intel {



// ================================================================================================
// Register-resident forward pass.  A warp owns 16 tokens of a session for the whole stack: its rows of X, Q,
// the attention probabilities, the attention output, the FFN hidden and the pre-LN sum never leave registers.
// The only data shared between the warps of a session are the K and V rows, published once per layer as
// pre-split TF32 hi/lo planes in shared memory.  Every accumulator tile (rows g, g+8; columns 2t, 2t+1) is
// turned into the A operand of the next product without a shuffle: the MMA k index is a free permutation as
// long as A and B agree, so k-slot t is mapped to column 2t and slot t+4 to column 2t+1 of each 8-wide block
// and the B fragments (weights, K rows, V^T rows) are read as one 8-byte load at [n = g][k = 2t].  Row strides
// of the planes are 8 or 24 (mod 32) words, which makes those loads bank-conflict free.
static const int WS = TD + 8;            // row stride of the weight and key planes

template <int MT>
struct RegTrunk {
    static constexpr int TP = 16 * MT;                  // padded tokens = 16 per warp
    static constexpr int NKT = 2 * MT;                  // key tiles of 8
    static constexpr int VS = TP + 8;                   // V^T plane stride
    static constexpr int WPL = TD * WS;                 // one weight plane
    static constexpr int off_wh = 0;                    // wq wk wv w1 w2, hi planes
    static constexpr int off_wl = 5 * WPL;              // lo planes
    static constexpr int off_vec = 10 * WPL;            // b1 b2 lnw lnb (fp32)
    static constexpr int off_sess = off_vec + 4 * TD;
    static constexpr int KPL = TP * WS, VPL = TD * VS;
    static constexpr int sess_words = 2 * KPL + 2 * VPL;    // K hi | K lo | V^T hi | V^T lo
    static constexpr size_t fwd_bytes(int sessions) { return (size_t)(off_sess + sessions * sess_words) * 4; }
};

__device__ __forceinline__ void stage_weights_split(uint32_t* sm, const TrunkArgs& a, int wpl, int off_wl, int off_vec) {
    const float* src[5] = {a.wq, a.wk, a.wv, a.w1, a.w2};
    for (int m = 0; m < 5; ++m)
        for (int e = threadIdx.x; e < TD * TD; e += blockDim.x) {
            uint32_t h, l;
            split_tf32(src[m][e], h, l);
            sm[m * wpl + (e / TD) * WS + (e % TD)] = h;
            sm[off_wl + m * wpl + (e / TD) * WS + (e % TD)] = l;
        }
    float* v = reinterpret_cast<float*>(sm) + off_vec;
    for (int e = threadIdx.x; e < TD; e += blockDim.x) {
        v[e] = a.b1[e]; v[TD + e] = a.b2[e]; v[2 * TD + e] = a.lnw[e]; v[3 * TD + e] = a.lnb[e];
    }
}

// accumulator tile -> pre-split A fragment of the k-step covering the same 8 columns
__device__ __forceinline__ void c_to_a(const float (&c)[4], uint32_t (&h)[4], uint32_t (&l)[4]) {
    split_tf32(c[0], h[0], l[0]);    // a0 = (g,   slot t)   <- column 2t
    split_tf32(c[2], h[1], l[1]);    // a1 = (g+8, slot t)
    split_tf32(c[1], h[2], l[2]);    // a2 = (g,   slot t+4) <- column 2t+1
    split_tf32(c[3], h[3], l[3]);    // a3 = (g+8, slot t+4)
}

// acc (16 x 8 NT) += A (16 x 8 KS, pre-split fragments) * B,  B(k, n) = plane[n * stride + k] (pre-split planes,
// already offset to the first n row / k column).  The small cross terms go to their own accumulators: shorter
// dependent MMA chains, and they are summed before they meet the large term.
template <int NT, int KS>
__device__ __forceinline__ void mma_planes(float (&acc)[NT][4], const uint32_t (&ah)[KS][4], const uint32_t (&al)[KS][4],
                                           const uint32_t* __restrict__ Bh, const uint32_t* __restrict__ Bl, int stride, int lane) {
    const int off = (lane >> 2) * stride + 2 * (lane & 3);
    float low[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) low[j][c] = 0.f;
#pragma unroll
    for (int s = 0; s < KS; ++s) {
        uint32_t bh[NT][2], bl[NT][2];
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            const uint2 h = *reinterpret_cast<const uint2*>(Bh + off + j * 8 * stride + s * 8);
            const uint2 l = *reinterpret_cast<const uint2*>(Bl + off + j * 8 * stride + s * 8);
            bh[j][0] = h.x; bh[j][1] = h.y; bl[j][0] = l.x; bl[j][1] = l.y;
        }
#pragma unroll
        for (int j = 0; j < NT; ++j) mma_tf32(low[j], al[s], bh[j]);
#pragma unroll
        for (int j = 0; j < NT; ++j) mma_tf32(low[j], ah[s], bl[j]);
#pragma unroll
        for (int j = 0; j < NT; ++j) mma_tf32(acc[j], ah[s], bh[j]);
    }
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[j][c] += low[j][c];
}

__device__ __forceinline__ float quad_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}
__device__ __forceinline__ float quad_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
    return v;
}

// attention of one head for the warp's 16 query rows: probabilities p (normalised, accumulator layout over the
// key tiles) and the head's output columns o.  q: the head's DK/8 accumulator tiles of Q.
template <int MT, int DK>
__device__ __forceinline__ void head_forward(const float (&q)[DK / 8][4], const uint32_t* Kh, const uint32_t* Kl,
                                             const uint32_t* Vh, const uint32_t* Vl, int ho, int L, int nkt, int lane,
                                             float (&p)[2 * MT][4], float (&o)[DK / 8][4]) {
    constexpr int NKT = 2 * MT, KS = DK / 8, VS = RegTrunk<MT>::VS;
    const int g = lane >> 2, t = lane & 3;
    const float scale = 1.0f / sqrtf((float)DK);
    uint32_t qh[KS][4], ql[KS][4];
#pragma unroll
    for (int s = 0; s < KS; ++s) c_to_a(q[s], qh[s], ql[s]);
#pragma unroll
    for (int j = 0; j < NKT; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) p[j][c] = 0.f;
    // S = Q_h K_h^T: B(k = channel, n = key) = K[key][ho + channel]
    {
        const int off = g * WS + ho + 2 * t;
#pragma unroll
        for (int s = 0; s < KS; ++s) {
#pragma unroll
            for (int j = 0; j < NKT; ++j) {
                if (j < nkt) {
                    const uint2 h = *reinterpret_cast<const uint2*>(Kh + off + j * 8 * WS + s * 8);
                    const uint2 l = *reinterpret_cast<const uint2*>(Kl + off + j * 8 * WS + s * 8);
                    const uint32_t bh[2] = {h.x, h.y}, bl[2] = {l.x, l.y};
                    mma_tf32(p[j], ql[s], bh);
                    mma_tf32(p[j], qh[s], bl);
                    mma_tf32(p[j], qh[s], bh);
                }
            }
        }
    }
    // softmax over the L live keys (list pads are live keys, IntEL.py:182-197; slots >= L do not exist)
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < NKT; ++j) {
        if (j < nkt) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const bool live = j * 8 + 2 * t + c < L;
                p[j][c] = live ? p[j][c] * scale : -INFINITY;
                p[j][2 + c] = live ? p[j][2 + c] * scale : -INFINITY;
                m0 = fmaxf(m0, p[j][c]);
                m1 = fmaxf(m1, p[j][2 + c]);
            }
        }
    }
    m0 = quad_max(m0);
    m1 = quad_max(m1);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < NKT; ++j) {
        if (j < nkt) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                p[j][c] = expf(p[j][c] - m0);
                p[j][2 + c] = expf(p[j][2 + c] - m1);
                s0 += p[j][c];
                s1 += p[j][2 + c];
            }
        }
    }
    const float i0 = 1.0f / quad_sum(s0), i1 = 1.0f / quad_sum(s1);
#pragma unroll
    for (int j = 0; j < NKT; ++j) {
        p[j][0] *= i0; p[j][1] *= i0; p[j][2] *= i1; p[j][3] *= i1;
    }
    // O_h = P V_h: k = key (tile j is k-step j), B(k = key, n = channel) = V^T[ho + channel][key]; even and odd
    // key tiles and the cross terms accumulate separately (four short chains per output tile)
    float oe[KS][4], oo[KS][4], ol[KS][4];
#pragma unroll
    for (int n = 0; n < KS; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) { oe[n][c] = 0.f; oo[n][c] = 0.f; ol[n][c] = 0.f; }
    {
        const int off = (ho + g) * VS + 2 * t;
#pragma unroll
        for (int j = 0; j < NKT; ++j) {
            if (j < nkt) {
                uint32_t ph[4], pl[4];
                c_to_a(p[j], ph, pl);
#pragma unroll
                for (int n = 0; n < KS; ++n) {
                    const uint2 h = *reinterpret_cast<const uint2*>(Vh + off + n * 8 * VS + j * 8);
                    const uint2 l = *reinterpret_cast<const uint2*>(Vl + off + n * 8 * VS + j * 8);
                    const uint32_t bh[2] = {h.x, h.y}, bl[2] = {l.x, l.y};
                    mma_tf32(ol[n], pl, bh);
                    mma_tf32(ol[n], ph, bl);
                    if (j & 1) mma_tf32(oo[n], ph, bh);
                    else mma_tf32(oe[n], ph, bh);
                }
            }
        }
    }
#pragma unroll
    for (int n = 0; n < KS; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) o[n][c] = (oe[n][c] + oo[n][c]) + ol[n][c];
}

template <int MT, int DK, int NS>
__global__ void __launch_bounds__(32 * MT * NS) trunk_fwd_kernel(TrunkArgs a) {
    using RT = RegTrunk<MT>;
    constexpr int HEADS = TD / DK, KS = DK / 8;
    DYN_SMEM(uint32_t, sm);
    const uint32_t* Wh = sm + RT::off_wh;
    const uint32_t* Wl = sm + RT::off_wl;
    const float* vec = reinterpret_cast<const float*>(sm) + RT::off_vec;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = warp / MT, mt = warp % MT;
    const int g = lane >> 2, t = lane & 3;
    uint32_t* Kh = sm + RT::off_sess + slot * RT::sess_words;
    uint32_t* Kl = Kh + RT::KPL;
    uint32_t* Vh = Kl + RT::KPL;
    uint32_t* Vl = Vh + RT::VPL;
    stage_weights_split(sm, a, RT::WPL, RT::off_wl, RT::off_vec);
    __syncthreads();
    const int L = a.L, nkt = (L + 7) >> 3;
    const int r0 = mt * 16 + g, r1 = r0 + 8;                    // this lane's two tokens
    const bool live0 = r0 < L, live1 = r1 < L;

    for (int64_t b = (int64_t)blockIdx.x * NS + slot; b < a.B; b += (int64_t)gridDim.x * NS) {
        const int64_t row0 = b * L;
        float x[4][4];                                          // layer input / output, accumulator layout
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 lo = live0 ? *reinterpret_cast<const float2*>(a.X[0] + (row0 + r0) * TD + j * 8 + 2 * t) : make_float2(0.f, 0.f);
            const float2 hi = live1 ? *reinterpret_cast<const float2*>(a.X[0] + (row0 + r1) * TD + j * 8 + 2 * t) : make_float2(0.f, 0.f);
            x[j][0] = lo.x; x[j][1] = lo.y; x[j][2] = hi.x; x[j][3] = hi.y;
        }
        for (int l = 0; l < a.layers; ++l) {
            float q[4][4];
            {
                uint32_t xh[4][4], xl[4][4];
#pragma unroll
                for (int s = 0; s < 4; ++s) c_to_a(x[s], xh[s], xl[s]);
                float kv[4][4];
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) { q[j][c] = 0.f; kv[j][c] = 0.f; }
                mma_planes<4, 4>(q, xh, xl, Wh + 0 * RT::WPL, Wl + 0 * RT::WPL, WS, lane);
                mma_planes<4, 4>(kv, xh, xl, Wh + 1 * RT::WPL, Wl + 1 * RT::WPL, WS, lane);
                if (MT > 1) bar_sync(1 + slot, 32 * MT);        // every warp is done with the previous K / V planes
                else __syncwarp();
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t h[4], lw[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) split_tf32(kv[j][c], h[c], lw[c]);
                    *reinterpret_cast<uint2*>(Kh + r0 * WS + j * 8 + 2 * t) = make_uint2(h[0], h[1]);
                    *reinterpret_cast<uint2*>(Kl + r0 * WS + j * 8 + 2 * t) = make_uint2(lw[0], lw[1]);
                    *reinterpret_cast<uint2*>(Kh + r1 * WS + j * 8 + 2 * t) = make_uint2(h[2], h[3]);
                    *reinterpret_cast<uint2*>(Kl + r1 * WS + j * 8 + 2 * t) = make_uint2(lw[2], lw[3]);
                }
                if (a.save) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float* d0 = a.QKV[l] + (row0 + r0) * 3 * TD + j * 8 + 2 * t;
                        float* d1 = a.QKV[l] + (row0 + r1) * 3 * TD + j * 8 + 2 * t;
                        if (live0) { *reinterpret_cast<float2*>(d0) = make_float2(q[j][0], q[j][1]); *reinterpret_cast<float2*>(d0 + TD) = make_float2(kv[j][0], kv[j][1]); }
                        if (live1) { *reinterpret_cast<float2*>(d1) = make_float2(q[j][2], q[j][3]); *reinterpret_cast<float2*>(d1 + TD) = make_float2(kv[j][2], kv[j][3]); }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) kv[j][c] = 0.f;
                mma_planes<4, 4>(kv, xh, xl, Wh + 2 * RT::WPL, Wl + 2 * RT::WPL, WS, lane);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t h[4], lw[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) split_tf32(kv[j][c], h[c], lw[c]);
                    const int c0 = j * 8 + 2 * t;
                    Vh[c0 * RT::VS + r0] = h[0]; Vh[(c0 + 1) * RT::VS + r0] = h[1];
                    Vh[c0 * RT::VS + r1] = h[2]; Vh[(c0 + 1) * RT::VS + r1] = h[3];
                    Vl[c0 * RT::VS + r0] = lw[0]; Vl[(c0 + 1) * RT::VS + r0] = lw[1];
                    Vl[c0 * RT::VS + r1] = lw[2]; Vl[(c0 + 1) * RT::VS + r1] = lw[3];
                }
                if (a.save) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (live0) *reinterpret_cast<float2*>(a.QKV[l] + (row0 + r0) * 3 * TD + 2 * TD + j * 8 + 2 * t) = make_float2(kv[j][0], kv[j][1]);
                        if (live1) *reinterpret_cast<float2*>(a.QKV[l] + (row0 + r1) * 3 * TD + 2 * TD + j * 8 + 2 * t) = make_float2(kv[j][2], kv[j][3]);
                    }
                }
            }
            if (MT > 1) bar_sync(1 + slot, 32 * MT);            // K / V of all tokens are visible
            else __syncwarp();
            float att[4][4];                                    // attention output, all heads
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                float p[2 * MT][4], o[KS][4], qq[KS][4];
#pragma unroll
                for (int s = 0; s < KS; ++s)
#pragma unroll
                    for (int c = 0; c < 4; ++c) qq[s][c] = q[hd * KS + s][c];
                head_forward<MT, DK>(qq, Kh, Kl, Vh, Vl, hd * DK, L, nkt, lane, p, o);
#pragma unroll
                for (int s = 0; s < KS; ++s)
#pragma unroll
                    for (int c = 0; c < 4; ++c) att[hd * KS + s][c] = o[s][c];
            }
            // FFN: U = A W1^T + b1,  Z = dropout(relu(U) W2^T + b2) + X,  X' = LayerNorm(Z)
            float u[4][4], z[4][4];
            {
                uint32_t ah[4][4], al[4][4];
#pragma unroll
                for (int s = 0; s < 4; ++s) c_to_a(att[s], ah[s], al[s]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 bb = *reinterpret_cast<const float2*>(vec + j * 8 + 2 * t);
                    u[j][0] = bb.x; u[j][1] = bb.y; u[j][2] = bb.x; u[j][3] = bb.y;
                }
                mma_planes<4, 4>(u, ah, al, Wh + 3 * RT::WPL, Wl + 3 * RT::WPL, WS, lane);
            }
            {
                uint32_t uh[4][4], ul[4][4];
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float r[4] = {fmaxf(u[s][0], 0.f), fmaxf(u[s][1], 0.f), fmaxf(u[s][2], 0.f), fmaxf(u[s][3], 0.f)};
                    c_to_a(r, uh[s], ul[s]);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 bb = *reinterpret_cast<const float2*>(vec + TD + j * 8 + 2 * t);
                    z[j][0] = bb.x; z[j][1] = bb.y; z[j][2] = bb.x; z[j][3] = bb.y;
                }
                mma_planes<4, 4>(z, uh, ul, Wh + 4 * RT::WPL, Wl + 4 * RT::WPL, WS, lane);
            }
            const Dropout& dr = a.drop[l];
            float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int col = j * 8 + 2 * t + c;
                    // dropout acts on the FFN output before the residual (IntEL.py:187-188)
                    z[j][c] = z[j][c] * dropout_scale(dr, row0 + r0, col, TD) + x[j][c];
                    z[j][2 + c] = z[j][2 + c] * dropout_scale(dr, row0 + r1, col, TD) + x[j][2 + c];
                    sum0 += z[j][c];
                    sum1 += z[j][2 + c];
                }
            }
            const float mean0 = quad_sum(sum0) * (1.0f / TD), mean1 = quad_sum(sum1) * (1.0f / TD);
            float v0 = 0.f, v1 = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const float d0 = z[j][c] - mean0, d1 = z[j][2 + c] - mean1;
                    v0 = fmaf(d0, d0, v0);
                    v1 = fmaf(d1, d1, v1);
                }
            const float rstd0 = rsqrtf(quad_sum(v0) * (1.0f / TD) + 1e-5f), rstd1 = rsqrtf(quad_sum(v1) * (1.0f / TD) + 1e-5f);
            if (a.save) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int64_t o0 = (row0 + r0) * TD + j * 8 + 2 * t, o1 = (row0 + r1) * TD + j * 8 + 2 * t;
                    if (live0) {
                        *reinterpret_cast<float2*>(a.A[l] + o0) = make_float2(att[j][0], att[j][1]);
                        *reinterpret_cast<float2*>(a.U[l] + o0) = make_float2(u[j][0], u[j][1]);
                        *reinterpret_cast<float2*>(a.Z[l] + o0) = make_float2(z[j][0], z[j][1]);
                    }
                    if (live1) {
                        *reinterpret_cast<float2*>(a.A[l] + o1) = make_float2(att[j][2], att[j][3]);
                        *reinterpret_cast<float2*>(a.U[l] + o1) = make_float2(u[j][2], u[j][3]);
                        *reinterpret_cast<float2*>(a.Z[l] + o1) = make_float2(z[j][2], z[j][3]);
                    }
                }
                if (t == 0) {
                    if (live0) *reinterpret_cast<float2*>(a.ST[l] + (row0 + r0) * 2) = make_float2(mean0, rstd0);
                    if (live1) *reinterpret_cast<float2*>(a.ST[l] + (row0 + r1) * 2) = make_float2(mean1, rstd1);
                }
            }
            float* out = a.X[l + 1];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 gw = *reinterpret_cast<const float2*>(vec + 2 * TD + j * 8 + 2 * t);
                const float2 gb = *reinterpret_cast<const float2*>(vec + 3 * TD + j * 8 + 2 * t);
                x[j][0] = (z[j][0] - mean0) * rstd0 * gw.x + gb.x;
                x[j][1] = (z[j][1] - mean0) * rstd0 * gw.y + gb.y;
                x[j][2] = (z[j][2] - mean1) * rstd1 * gw.x + gb.x;
                x[j][3] = (z[j][3] - mean1) * rstd1 * gw.y + gb.y;
                if (!live0) { x[j][0] = 0.f; x[j][1] = 0.f; }       // pad tokens stay zero like the padded input rows
                if (!live1) { x[j][2] = 0.f; x[j][3] = 0.f; }
                if (a.save || l == a.layers - 1) {
                    if (live0) *reinterpret_cast<float2*>(out + (row0 + r0) * TD + j * 8 + 2 * t) = make_float2(x[j][0], x[j][1]);
                    if (live1) *reinterpret_cast<float2*>(out + (row0 + r1) * TD + j * 8 + 2 * t) = make_float2(x[j][2], x[j][3]);
                }
            }
        }
    }
}

// ================================================================================================
// Register-resident backward pass.  Four warps per session, NS = 2 or 3 sessions per CTA (each with its own named
// barrier).  Token-local work (LayerNorm, FFN and projection input gradients, the attention rows of a query
// block) is done by the warp that owns the 16 tokens, on accumulator-layout registers as in the forward kernel.
// Products that contract over the tokens of a session go through shared-memory tiles:
//   region B: K | V | Q | dA tiles          -> S, dP, dQ (row-local), dK = dS^T Q, dV = P^T dA (key-local)
//   region C: first dF | dU tiles           -> dW2 = dF^T relu(U), dW1 = dU^T A     (B operands read from HBM/L1)
//             then P | dS of one head, last dQ | dK | dV tiles -> dWq/dWk/dWv = d{Q,K,V}^T X
// Weight-gradient tiles are owned by fixed warps (2 tiles per matrix and warp) and live across all sessions of the
// CTA; each session's contribution is summed from zero and folded in with a rounded add.  They and the dQ | dK | dV
// rows of the head loop are parked in tensor memory (Park below): at 168 registers three sessions (12 warps) fit an
// SM, which hides more of the dependent-MMA latency this kernel waits on than 8 warps did.
static const int BWD_WPS = 4;
static const int kMaxSmemBytes = 227 * 1024;

struct BwdPlan {
    int nkt, rows, ds, tile, ps, region_c, sess, off_cs, off_sess, total;     // in 4-byte words
    bool fits() const { return (size_t)total * 4 <= (size_t)kMaxSmemBytes; }
};
__host__ __device__ inline BwdPlan bwd_plan(int L, int ns) {
    BwdPlan p;
    p.nkt = (L + 7) >> 3;
    p.rows = 8 * p.nkt;
    p.ds = (p.nkt & 1) ? 8 * p.nkt : 8 * p.nkt + 8;        // row stride of P / dS: an odd multiple of 8 words
    p.tile = p.rows * WS;
    p.ps = p.rows * p.ds;
    p.region_c = 2 * p.ps > 3 * p.tile ? 2 * p.ps : 3 * p.tile;
    p.sess = 4 * p.tile + p.region_c;
    p.off_cs = 5 * TD * WS;                                  // after the five transposed weight planes
    p.off_sess = p.off_cs + ns * BWD_WPS * 4 * TD;
    p.total = p.off_sess + ns * p.sess;
    return p;
}

// Per-thread values that live across much of the kernel but are touched rarely, parked in the thread's own lane of
// tensor memory (the warp's 32-lane quarter): eight columns move per access, as two accumulator tiles.  tcgen05.ld /
// st are warp-collective, so every access is warp-uniform.  The emulator has no tensor memory and keeps them in
// registers, so that it runs the same kernel body.
struct Park {
    static constexpr int PW = 0, DQ = 40, DK = 56, DV = 72, COLS = 88;   // 5 weight-gradient tile pairs, dQ | dK | dV rows
#ifdef INTEL_EMU
    float r[COLS];
    void get(float (*v)[4], int col) const {
        for (int i = 0; i < 8; ++i) v[i >> 2][i & 3] = r[col + i];
    }
    void put(const float (*v)[4], int col) {
        for (int i = 0; i < 8; ++i) r[col + i] = v[i >> 2][i & 3];
    }
#else
    uint32_t base;                                                        // lane quarter + this warp's first column
    __device__ __forceinline__ void get(float (*v)[4], int col) const {
        uint32_t u[8];
        tc05::wait_st();
        tc05::ld8(base + col, u);
        tc05::wait_ld();
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i >> 2][i & 3] = __uint_as_float(u[i]);
    }
    __device__ __forceinline__ void put(const float (*v)[4], int col) {
        uint32_t u[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) u[i] = __float_as_uint(v[i >> 2][i & 3]);
        tc05::st8(base + col, u);
    }
#endif
};

// acc (16 x 8 NT) += A * B with B(k, n) = B[n * stride + k] read as fp32 and split here; tiles >= nlive are skipped
template <int NT, int KS>
__device__ __forceinline__ void mma_raw(float (&acc)[NT][4], const uint32_t (&ah)[KS][4], const uint32_t (&al)[KS][4],
                                        const float* __restrict__ B, int stride, int nlive, int lane) {
    const int off = (lane >> 2) * stride + 2 * (lane & 3);
#pragma unroll
    for (int j = 0; j < NT; ++j) {                  // tile by tile: one small-term accumulator live instead of NT
        if (j < nlive) {
            float low[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int s = 0; s < KS; ++s) {
                const float2 v = *reinterpret_cast<const float2*>(B + off + j * 8 * stride + s * 8);
                uint32_t bh[2], bl[2];
                split_tf32(v.x, bh[0], bl[0]);
                split_tf32(v.y, bh[1], bl[1]);
                mma_tf32(low, al[s], bh);
                mma_tf32(low, ah[s], bl);
                mma_tf32(acc[j], ah[s], bh);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[j][c] += low[c];
        }
    }
}

// rows r0 / r1 of an accumulator-layout [16 x 32] block -> fp32 tile [rows][WS]
__device__ __forceinline__ void put_tile(float* T, const float (&v)[4][4], int r0, int r1, int rows, int t) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (r0 < rows) *reinterpret_cast<float2*>(T + r0 * WS + j * 8 + 2 * t) = make_float2(v[j][0], v[j][1]);
        if (r1 < rows) *reinterpret_cast<float2*>(T + r1 * WS + j * 8 + 2 * t) = make_float2(v[j][2], v[j][3]);
    }
}
// rows r0 / r1 of a row-major [*, ld] global tensor -> accumulator layout (dead rows read as zero)
__device__ __forceinline__ void get_rows(float (&v)[4][4], const float* __restrict__ src, int64_t ld, int64_t g0, int64_t g1,
                                         bool live0, bool live1, int t) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 lo = live0 ? *reinterpret_cast<const float2*>(src + g0 * ld + j * 8 + 2 * t) : make_float2(0.f, 0.f);
        const float2 hi = live1 ? *reinterpret_cast<const float2*>(src + g1 * ld + j * 8 + 2 * t) : make_float2(0.f, 0.f);
        v[j][0] = lo.x; v[j][1] = lo.y; v[j][2] = hi.x; v[j][3] = hi.y;
    }
}
// column sums of an accumulator-layout block over the warp's 16 rows, added to a warp-private shared vector
__device__ __forceinline__ void colsum_rows(float* slot, const float (&v)[4][4], int lane) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float x = v[j][c] + v[j][2 + c];
            x += __shfl_xor_sync(0xffffffffu, x, 4);
            x += __shfl_xor_sync(0xffffffffu, x, 8);
            x += __shfl_xor_sync(0xffffffffu, x, 16);
            if ((lane >> 2) == 0) slot[j * 8 + 2 * (lane & 3) + c] += x;
        }
}

// rows r0 / r1 of a fp32 tile [rows][WS], columns col .. col + 7 -> accumulator layout (rows >= rows read as zero)
__device__ __forceinline__ void get_tile(float (&v)[4], const float* T, int r0, int r1, int rows, int col, int t) {
    const float2 lo = r0 < rows ? *reinterpret_cast<const float2*>(T + r0 * WS + col + 2 * t) : make_float2(0.f, 0.f);
    const float2 hi = r1 < rows ? *reinterpret_cast<const float2*>(T + r1 * WS + col + 2 * t) : make_float2(0.f, 0.f);
    v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
}

// parked tile pair pw + 8 a (this warp's two 16x8 tiles of a 32x32 weight gradient) += T[a]^T B over the session's
// tokens, for NA gradient tiles that share the B operand.  T[a]: shared tile [rows][WS] (m = T column), B: global rows
// of the session [L][ldb] (n = B column), optional relu.  All B fragments are fetched before the first MMA so that the
// global-memory latency is paid once, not once per k-step.
template <int NA, int NKT, bool RELU>
__device__ __forceinline__ void wgrad_tiles(Park& park, int pw, const float* const (&T)[NA], const float* __restrict__ Bg, int ldb,
                                            int L, int nkt, int w, int lane) {
    const int g = lane >> 2, t = lane & 3;
    const int m0 = (w & 1) * 16 + g, n0 = (w >> 1) * 16 + g;
    float bv[NKT][2][2];
#pragma unroll
    for (int s = 0; s < NKT; ++s) {
        const int k0 = 8 * s + t, k1 = k0 + 4;
#pragma unroll
        for (int n = 0; n < 2; ++n) {
            float b0 = (s < nkt && k0 < L) ? Bg[(int64_t)k0 * ldb + n0 + 8 * n] : 0.f;
            float b1 = (s < nkt && k1 < L) ? Bg[(int64_t)k1 * ldb + n0 + 8 * n] : 0.f;
            if (RELU) { b0 = fmaxf(b0, 0.f); b1 = fmaxf(b1, 0.f); }
            bv[s][n][0] = b0;
            bv[s][n][1] = b1;
        }
    }
#pragma unroll
    for (int a = 0; a < NA; ++a) {
        float part[2][4];
#pragma unroll
        for (int n = 0; n < 2; ++n)
#pragma unroll
            for (int c = 0; c < 4; ++c) part[n][c] = 0.f;
#pragma unroll
        for (int s = 0; s < NKT; ++s) {
            if (s < nkt) {
                const int k0 = 8 * s + t, k1 = k0 + 4;
                const float* Ta = T[a];
                const float af[4] = {Ta[k0 * WS + m0], Ta[k0 * WS + m0 + 8], Ta[k1 * WS + m0], Ta[k1 * WS + m0 + 8]};
#pragma unroll
                for (int n = 0; n < 2; ++n) mma_3xtf32(part[n], af, bv[s][n]);
            }
        }
        float acc[2][4];
        park.get(acc, pw + 8 * a);
#pragma unroll
        for (int n = 0; n < 2; ++n)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[n][c] += part[n][c];
        park.put(acc, pw + 8 * a);
    }
}

template <int MT, int DK, int NS>
__global__ void __launch_bounds__(32 * NS * BWD_WPS, 1) trunk_bwd_kernel(TrunkArgs a) {
    constexpr int HEADS = TD / DK, KS = DK / 8, NKT = 2 * MT;
    static_assert(KS % 2 == 0, "dQ | dK | dV rows are parked in pairs of accumulator tiles");
    DYN_SMEM(float, sm);
    const int L = a.L;
    const BwdPlan pl = bwd_plan(L, NS);
    const int nkt = pl.nkt, rows = pl.rows, DS = pl.ds;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = warp / BWD_WPS, w = warp % BWD_WPS;
    const int g = lane >> 2, t = lane & 3;
    const float scale = 1.0f / sqrtf((float)DK);
    const float* WT = sm;                                   // transposed weights: WT[m][k_in * WS + n_out]
    float* cs = sm + pl.off_cs + warp * 4 * TD;             // this warp's column sums: db1 | db2 | dlnw | dlnb
    float* sess = sm + pl.off_sess + slot * pl.sess;
    float* T_K = sess;
    float* T_V = T_K + pl.tile;
    float* T_Q = T_V + pl.tile;
    float* T_dA = T_Q + pl.tile;
    float* Ps = T_dA + pl.tile;                             // region C
    float* Ds = Ps + pl.ps;
    float* T_dF = Ps;
    float* T_dU = T_dF + pl.tile;
    float* T_dQ = Ps;
    float* T_dK = T_dQ + pl.tile;
    float* T_dV = T_dK + pl.tile;
    {
        const float* src[5] = {a.wq, a.wk, a.wv, a.w1, a.w2};
        for (int m = 0; m < 5; ++m)
            for (int e = threadIdx.x; e < TD * TD; e += blockDim.x) sm[m * TD * WS + (e % TD) * WS + (e / TD)] = src[m][e];
        for (int e = threadIdx.x; e < NS * BWD_WPS * 4 * TD; e += blockDim.x) sm[pl.off_cs + e] = 0.f;
    }
    // tensor memory: the warps w of all sessions share lane quarter w, 128 columns per session
    constexpr uint32_t TMEM_COLS = NS * 128 <= 256 ? 256 : 512;
    static_assert(Park::COLS <= 128 && NS * 128 <= 512, "parked columns exceed tensor memory");
    Park park;
#ifdef INTEL_EMU
    __syncthreads();
#else
    __shared__ uint32_t tmem_slot;
    if (warp == 0) tc05::tmem_alloc(&tmem_slot, TMEM_COLS);
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    park.base = tmem_slot + ((uint32_t)(w * 32) << 16) + (uint32_t)(slot * 128);
#endif
    const float* lnw = a.lnw;
    {
        const float zero[2][4] = {};                        // weight-gradient tiles: w2 w1 wq wk wv
#pragma unroll
        for (int m = 0; m < 5; ++m) park.put(zero, Park::PW + 8 * m);
    }
    const bool rowwarp = w < MT;                            // owns tokens 16 w .. 16 w + 15
    const int r0 = w * 16 + g, r1 = r0 + 8;
    const bool live0 = rowwarp && r0 < L, live1 = rowwarp && r1 < L;
    const int bar = 1 + slot;

    for (int64_t b = (int64_t)blockIdx.x * NS + slot; b < a.B; b += (int64_t)gridDim.x * NS) {
        const int64_t row0 = b * L;
        float gx[4][4];                                     // d loss / d (layer output) of the warp's tokens
        get_rows(gx, a.dX, TD, row0 + r0, row0 + r1, live0, live1, t);
        for (int l = a.layers - 1; l >= 0; --l) {
            float df[4][4];
            if (rowwarp) {
                // ---- LayerNorm backward: gx <- dZ ----
                {
                    float z[4][4];
                    get_rows(z, a.Z[l], TD, row0 + r0, row0 + r1, live0, live1, t);
                    const float2 st0 = live0 ? *reinterpret_cast<const float2*>(a.ST[l] + (row0 + r0) * 2) : make_float2(0.f, 0.f);
                    const float2 st1 = live1 ? *reinterpret_cast<const float2*>(a.ST[l] + (row0 + r1) * 2) : make_float2(0.f, 0.f);
                    float dgam[4][4], s1a = 0.f, s2a = 0.f, s1b = 0.f, s2b = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 gw = *reinterpret_cast<const float2*>(lnw + j * 8 + 2 * t);
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            const float wv = c ? gw.y : gw.x;
                            const float xa = (z[j][c] - st0.x) * st0.y, xb = (z[j][2 + c] - st1.x) * st1.y;
                            const float ga = gx[j][c] * wv, gb = gx[j][2 + c] * wv;
                            dgam[j][c] = gx[j][c] * xa;
                            dgam[j][2 + c] = gx[j][2 + c] * xb;
                            s1a += ga; s2a = fmaf(ga, xa, s2a);
                            s1b += gb; s2b = fmaf(gb, xb, s2b);
                            z[j][c] = xa; z[j][2 + c] = xb;
                        }
                    }
                    colsum_rows(cs + 2 * TD, dgam, lane);
                    colsum_rows(cs + 3 * TD, gx, lane);
                    s1a = quad_sum(s1a) * (1.0f / TD); s2a = quad_sum(s2a) * (1.0f / TD);
                    s1b = quad_sum(s1b) * (1.0f / TD); s2b = quad_sum(s2b) * (1.0f / TD);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 gw = *reinterpret_cast<const float2*>(lnw + j * 8 + 2 * t);
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            const float wv = c ? gw.y : gw.x;
                            gx[j][c] = st0.y * (gx[j][c] * wv - s1a - z[j][c] * s2a);
                            gx[j][2 + c] = st1.y * (gx[j][2 + c] * wv - s1b - z[j][2 + c] * s2b);
                        }
                    }
                }
                // ---- FFN backward (token-local part): dF = dZ * dropout mask, dU = (dF W2) * (U > 0), dA = dU W1 ----
                const Dropout& dr = a.drop[l];
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int col = j * 8 + 2 * t + c;
                        df[j][c] = gx[j][c] * dropout_scale(dr, row0 + r0, col, TD);
                        df[j][2 + c] = gx[j][2 + c] * dropout_scale(dr, row0 + r1, col, TD);
                    }
            }
            bar_sync(bar, 32 * BWD_WPS);                                                   // s0: region C is read (dQ | dK | dV)
            if (rowwarp) {
                put_tile(T_dF, df, r0, r1, rows, t);
                colsum_rows(cs + TD, df, lane);
                float du[4][4];
                {
                    uint32_t fh[4][4], fl[4][4];
#pragma unroll
                    for (int s = 0; s < 4; ++s) c_to_a(df[s], fh[s], fl[s]);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) du[j][c] = 0.f;
                    mma_raw<4, 4>(du, fh, fl, WT + 4 * TD * WS, WS, 4, lane);
                    float u[4][4];
                    get_rows(u, a.U[l], TD, row0 + r0, row0 + r1, live0, live1, t);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) du[j][c] = u[j][c] > 0.f ? du[j][c] : 0.f;
                }
                put_tile(T_dU, du, r0, r1, rows, t);
                colsum_rows(cs, du, lane);
                {
                    uint32_t uh[4][4], ul[4][4];
                    float da[4][4];
#pragma unroll
                    for (int s = 0; s < 4; ++s) c_to_a(du[s], uh[s], ul[s]);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) da[j][c] = 0.f;
                    mma_raw<4, 4>(da, uh, ul, WT + 3 * TD * WS, WS, 4, lane);
                    put_tile(T_dA, da, r0, r1, rows, t);
                }
                // ---- the session's K, V, Q rows saved by the forward pass ----
                {
                    float kv[4][4];
                    get_rows(kv, a.QKV[l] + TD, 3 * TD, row0 + r0, row0 + r1, live0, live1, t);
                    put_tile(T_K, kv, r0, r1, rows, t);
                    get_rows(kv, a.QKV[l] + 2 * TD, 3 * TD, row0 + r0, row0 + r1, live0, live1, t);
                    put_tile(T_V, kv, r0, r1, rows, t);
                    get_rows(kv, a.QKV[l], 3 * TD, row0 + r0, row0 + r1, live0, live1, t);
                    put_tile(T_Q, kv, r0, r1, rows, t);
                }
            }
            bar_sync(bar, 32 * BWD_WPS);                                                   // s1: dF | dU and region B are complete
            {
                const float* const t2[1] = {T_dF};
                const float* const t1[1] = {T_dU};
                wgrad_tiles<1, NKT, true>(park, Park::PW + 0, t2, a.U[l] + row0 * TD, TD, L, nkt, w, lane);    // dW2 += dF^T relu(U)
                wgrad_tiles<1, NKT, false>(park, Park::PW + 8, t1, a.A[l] + row0 * TD, TD, L, nkt, w, lane);   // dW1 += dU^T A
            }
            bar_sync(bar, 32 * BWD_WPS);                                                   // s2: dF | dU are read, region C takes P | dS
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                const int ho = hd * DK;
                if (rowwarp) {
                    // ---- query rows of this warp: P, dP, dS, dQ_h ----
                    float p[NKT][4], dp[NKT][4];
#pragma unroll
                    for (int j = 0; j < NKT; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) { p[j][c] = 0.f; dp[j][c] = 0.f; }
                    {
                        uint32_t qh[KS][4], ql[KS][4];
#pragma unroll
                        for (int s = 0; s < KS; ++s) {
                            float f[4];
                            get_tile(f, T_Q, r0, r1, rows, ho + 8 * s, t);
                            c_to_a(f, qh[s], ql[s]);
                        }
                        mma_raw<NKT, KS>(p, qh, ql, T_K + ho, WS, nkt, lane);
#pragma unroll
                        for (int s = 0; s < KS; ++s) {
                            float f[4];
                            get_tile(f, T_dA, r0, r1, rows, ho + 8 * s, t);
                            c_to_a(f, qh[s], ql[s]);
                        }
                        mma_raw<NKT, KS>(dp, qh, ql, T_V + ho, WS, nkt, lane);
                    }
                    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
                    for (int j = 0; j < NKT; ++j) {
                        if (j < nkt) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                const bool live = j * 8 + 2 * t + c < L;
                                p[j][c] = live ? p[j][c] * scale : -INFINITY;
                                p[j][2 + c] = live ? p[j][2 + c] * scale : -INFINITY;
                                m0 = fmaxf(m0, p[j][c]);
                                m1 = fmaxf(m1, p[j][2 + c]);
                            }
                        }
                    }
                    m0 = quad_max(m0);
                    m1 = quad_max(m1);
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll
                    for (int j = 0; j < NKT; ++j) {
                        if (j < nkt) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                p[j][c] = expf(p[j][c] - m0);
                                p[j][2 + c] = expf(p[j][2 + c] - m1);
                                s0 += p[j][c];
                                s1 += p[j][2 + c];
                            }
                        }
                    }
                    const float i0 = 1.0f / quad_sum(s0), i1 = 1.0f / quad_sum(s1);
                    float d0 = 0.f, d1 = 0.f;
#pragma unroll
                    for (int j = 0; j < NKT; ++j) {
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            p[j][c] *= i0;
                            p[j][2 + c] *= i1;
                            d0 = fmaf(p[j][c], dp[j][c], d0);
                            d1 = fmaf(p[j][2 + c], dp[j][2 + c], d1);
                        }
                    }
                    d0 = quad_sum(d0);
                    d1 = quad_sum(d1);
#pragma unroll
                    for (int j = 0; j < NKT; ++j) {
                        if (j < nkt) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                dp[j][c] = p[j][c] * (dp[j][c] - d0) * scale;             // dS
                                dp[j][2 + c] = p[j][2 + c] * (dp[j][2 + c] - d1) * scale;
                            }
                            if (r0 < rows) {
                                *reinterpret_cast<float2*>(Ps + r0 * DS + j * 8 + 2 * t) = make_float2(p[j][0], p[j][1]);
                                *reinterpret_cast<float2*>(Ds + r0 * DS + j * 8 + 2 * t) = make_float2(dp[j][0], dp[j][1]);
                            }
                            if (r1 < rows) {
                                *reinterpret_cast<float2*>(Ps + r1 * DS + j * 8 + 2 * t) = make_float2(p[j][2], p[j][3]);
                                *reinterpret_cast<float2*>(Ds + r1 * DS + j * 8 + 2 * t) = make_float2(dp[j][2], dp[j][3]);
                            }
                        }
                    }
                    // dQ_h = dS K_h: k = key (tile j is k-step j), B(k = key, n = channel) = K[key][ho + channel]
                    float qe[KS][4], qo[KS][4];
#pragma unroll
                    for (int n = 0; n < KS; ++n)
#pragma unroll
                        for (int c = 0; c < 4; ++c) { qe[n][c] = 0.f; qo[n][c] = 0.f; }
#pragma unroll
                    for (int j = 0; j < NKT; ++j) {
                        if (j < nkt) {
                            const float af[4] = {dp[j][0], dp[j][2], dp[j][1], dp[j][3]};
#pragma unroll
                            for (int n = 0; n < KS; ++n) {
                                const float bf[2] = {T_K[(j * 8 + 2 * t) * WS + ho + n * 8 + g], T_K[(j * 8 + 2 * t + 1) * WS + ho + n * 8 + g]};
                                if (j & 1) mma_3xtf32(qo[n], af, bf);
                                else mma_3xtf32(qe[n], af, bf);
                            }
                        }
                    }
#pragma unroll
                    for (int n = 0; n < KS; n += 2) {
                        float d[2][4];
#pragma unroll
                        for (int c = 0; c < 4; ++c) { d[0][c] = qe[n][c] + qo[n][c]; d[1][c] = qe[n + 1][c] + qo[n + 1][c]; }
                        park.put(d, Park::DQ + 4 * (hd * KS + n));
                    }
                }
                bar_sync(bar, 32 * BWD_WPS);                                               // P / dS of every query row are visible
                if (rowwarp) {
                    // ---- keys 16 w .. 16 w + 15: dK_h = dS^T Q_h, dV_h = P^T dA_h (contraction over the query rows) ----
                    float ke[KS][4], ve[KS][4];
#pragma unroll
                    for (int n = 0; n < KS; ++n)
#pragma unroll
                        for (int c = 0; c < 4; ++c) { ke[n][c] = 0.f; ve[n][c] = 0.f; }
                    const int c0 = w * 16 + g, c1 = c0 + 8;
                    const bool in0 = c0 < rows, in1 = c1 < rows;
#pragma unroll 2
                    for (int s = 0; s < nkt; ++s) {
                        const int k0 = 8 * s + t, k1 = k0 + 4;
                        const float as[4] = {in0 ? Ds[k0 * DS + c0] : 0.f, in1 ? Ds[k0 * DS + c1] : 0.f, in0 ? Ds[k1 * DS + c0] : 0.f,
                                             in1 ? Ds[k1 * DS + c1] : 0.f};
                        const float ap[4] = {in0 ? Ps[k0 * DS + c0] : 0.f, in1 ? Ps[k0 * DS + c1] : 0.f, in0 ? Ps[k1 * DS + c0] : 0.f,
                                             in1 ? Ps[k1 * DS + c1] : 0.f};
#pragma unroll
                        for (int n = 0; n < KS; ++n) {
                            const float bq[2] = {T_Q[k0 * WS + ho + n * 8 + g], T_Q[k1 * WS + ho + n * 8 + g]};
                            const float ba[2] = {T_dA[k0 * WS + ho + n * 8 + g], T_dA[k1 * WS + ho + n * 8 + g]};
                            mma_3xtf32(ke[n], as, bq);
                            mma_3xtf32(ve[n], ap, ba);
                        }
                    }
#pragma unroll
                    for (int n = 0; n < KS; n += 2) {
                        const float dk[2][4] = {{ke[n][0], ke[n][1], ke[n][2], ke[n][3]}, {ke[n + 1][0], ke[n + 1][1], ke[n + 1][2], ke[n + 1][3]}};
                        const float dv[2][4] = {{ve[n][0], ve[n][1], ve[n][2], ve[n][3]}, {ve[n + 1][0], ve[n + 1][1], ve[n + 1][2], ve[n + 1][3]}};
                        park.put(dk, Park::DK + 4 * (hd * KS + n));
                        park.put(dv, Park::DV + 4 * (hd * KS + n));
                    }
                }
                bar_sync(bar, 32 * BWD_WPS);                                               // region C may be overwritten
            }
            if (rowwarp) {
                // ---- projections backward: dX = dQ Wq + dK Wk + dV Wv + dZ; dQ | dK | dV tiles for the weight gradients ----
                float* const td[3] = {T_dQ, T_dK, T_dV};
                const int col[3] = {Park::DQ, Park::DK, Park::DV};
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    float d[4][4];
                    park.get(d, col[m]);
                    park.get(d + 2, col[m] + 8);
                    put_tile(td[m], d, r0, r1, rows, t);
                    uint32_t fh[4][4], fl[4][4];
#pragma unroll
                    for (int s = 0; s < 4; ++s) c_to_a(d[s], fh[s], fl[s]);
                    mma_raw<4, 4>(gx, fh, fl, WT + m * TD * WS, WS, 4, lane);
                }
            }
            bar_sync(bar, 32 * BWD_WPS);                                                   // dQ | dK | dV tiles are complete
            {
                const float* const tq[3] = {T_dQ, T_dK, T_dV};
                wgrad_tiles<3, NKT, false>(park, Park::PW + 16, tq, a.X[l] + row0 * TD, TD, L, nkt, w, lane);   // dW{q,k,v} += d{Q,K,V}^T X
            }
        }
        if (rowwarp) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (live0) *reinterpret_cast<float2*>(a.dX + (row0 + r0) * TD + j * 8 + 2 * t) = make_float2(gx[j][0], gx[j][1]);
                if (live1) *reinterpret_cast<float2*>(a.dX + (row0 + r1) * TD + j * 8 + 2 * t) = make_float2(gx[j][2], gx[j][3]);
            }
        }
    }
    // ---- flush: weight-gradient tiles straight from tensor memory, vector gradients through the warp-private sums ----
    {
        float* dst[5] = {a.gw2, a.gw1, a.gwq, a.gwk, a.gwv};
        const int m0 = (w & 1) * 16 + g, n0 = (w >> 1) * 16 + 2 * t;
#pragma unroll
        for (int m = 0; m < 5; ++m) {
            float pw[2][4];
            park.get(pw, Park::PW + 8 * m);
#pragma unroll
            for (int n = 0; n < 2; ++n) {
                atomicAdd(dst[m] + m0 * TD + n0 + 8 * n, pw[n][0]);
                atomicAdd(dst[m] + m0 * TD + n0 + 8 * n + 1, pw[n][1]);
                atomicAdd(dst[m] + (m0 + 8) * TD + n0 + 8 * n, pw[n][2]);
                atomicAdd(dst[m] + (m0 + 8) * TD + n0 + 8 * n + 1, pw[n][3]);
            }
        }
    }
#ifndef INTEL_EMU
    tc05::fence_before();
#endif
    __syncthreads();
#ifndef INTEL_EMU
    if (warp == 0) {
        tc05::fence_after();
        tc05::tmem_free(tmem_slot, TMEM_COLS);
    }
#endif
    if (threadIdx.x < 4 * TD) {
        float v = 0.f;
        for (int ww = 0; ww < NS * BWD_WPS; ++ww) v += sm[pl.off_cs + ww * 4 * TD + threadIdx.x];
        float* dst = threadIdx.x < TD ? a.gb1 : (threadIdx.x < 2 * TD ? a.gb2 : (threadIdx.x < 3 * TD ? a.glnw : a.glnb));
        atomicAdd(dst + (threadIdx.x & (TD - 1)), v);
    }
}

bool trunk_supported(int64_t L, int d, int heads, int layers) {
    return d == TD && L >= 1 && L <= 64 && layers >= 1 && layers <= 8 && (heads == 1 || heads == 2);
}

static int g_sessions_per_cta = 4;
static int g_reserved_sms = 0, g_reserve_now = 0;
void trunk_reserve_sms(int n) { g_reserved_sms = n < 0 ? 0 : (n > 64 ? 64 : n); }
void trunk_reserve_apply(bool on) { g_reserve_now = on ? 1 : 0; }
void trunk_debug_sessions_per_cta(int n) { g_sessions_per_cta = n < 1 ? 1 : (n > 4 ? 4 : n); }

// algorithmic HBM bytes per token: the stack input (and dX in / out), and per layer the saved q|k|v (96), attention
// output, FFN hidden, pre-LN sum, layer output (32 each) and LN statistics (2) that the forward pass writes when it
// saves for backward and the backward pass reads back
static void trunk_account(const TrunkArgs& a, bool bwd, double& bytes, double& flops) {
    const double tok = (double)a.B * a.L;
    flops = tok * a.layers * (2.0 * 5 * TD * TD + 4.0 * a.L * TD) * (bwd ? 3.0 : 1.0);
    const double per_layer = (a.save || bwd) ? 4.0 * (3 * TD + 4 * TD + 2) : 0.0;
    bytes = tok * (4.0 * TD * (bwd ? 2 : 1) + per_layer * a.layers + ((a.save || bwd) ? 0.0 : 4.0 * TD));
}

template <int MT, int DK, int NS>
static int trunk_fwd_launch(const TrunkArgs& a, cudaStream_t s) {
    const size_t smem = RegTrunk<MT>::fwd_bytes(NS);
    const int per_sm = (int)(227 * 1024 / (smem + 1024));
    const unsigned grid = stream_grid((a.B + NS - 1) / NS, per_sm < 1 ? 1 : per_sm);
    auto k = trunk_fwd_kernel<MT, DK, NS>;
    ensure_smem(k, smem);
    LAUNCH(k, dim3(grid), dim3(32 * MT * NS), smem, s, a);
    double bytes, flops;
    trunk_account(a, false, bytes, flops);
    return check_launch("trunk_fwd", bytes, flops);
}

template <int MT, int DK>
static int trunk_fwd_sessions(const TrunkArgs& a, cudaStream_t s) {
    switch (g_sessions_per_cta) {
        case 1: return trunk_fwd_launch<MT, DK, 1>(a, s);
        case 2: return trunk_fwd_launch<MT, DK, 2>(a, s);
        case 3: return trunk_fwd_launch<MT, DK, 3>(a, s);
        default: return trunk_fwd_launch<MT, DK, 4>(a, s);
    }
}

template <int TP, int DK, int NS>
static int trunk_bwd_launch(const TrunkArgs& a, cudaStream_t s) {
    const size_t smem = (size_t)bwd_plan(a.L, NS).total * 4;
    unsigned grid = stream_grid((a.B + NS - 1) / NS, 1);
    if (g_reserve_now && grid > (unsigned)(kNumSMs - g_reserved_sms)) grid = (unsigned)(kNumSMs - g_reserved_sms);   // one CTA owns an SM
    auto k = trunk_bwd_kernel<TP / 16, DK, NS>;
    ensure_smem(k, smem);
    LAUNCH(k, dim3(grid), dim3(32 * NS * BWD_WPS), smem, s, a);
    double bytes, flops;
    trunk_account(a, true, bytes, flops);
    return check_launch("trunk_bwd", bytes, flops);
}

template <int TP, int DK>
static int trunk_launch(const TrunkArgs& a, bool bwd, cudaStream_t s) {
    if (!bwd) return trunk_fwd_sessions<TP / 16, DK>(a, s);
    // three sessions (12 warps) where their tiles fit in shared memory (L <= 56), two otherwise or when asked for
    if (g_sessions_per_cta >= 3 && bwd_plan(a.L, 3).fits()) return trunk_bwd_launch<TP, DK, 3>(a, s);
    return trunk_bwd_launch<TP, DK, 2>(a, s);
}

bool trunk_fwd_supported(int64_t L, int heads, int layers) {
    TrunkArgs a;
    memset(&a, 0, sizeof(a));
    a.L = (int)(L > 1 << 20 ? 1 << 20 : L); a.heads = heads; a.layers = layers;
    return trunk_tc_supported(a) || trunk_supported(L, TD, heads, layers);
}

int trunk_run(const TrunkArgs& a, bool bwd, cudaStream_t s) {
    if (a.B <= 0) return INTEL_OK;
    if (!bwd && trunk_tc_supported(a)) return trunk_tc_fwd(a, s);
    INTEL_REQUIRE(trunk_supported(a.L, TD, a.heads, a.layers), INTEL_ERR_UNSUPPORTED, "fused stack: unsupported shape");
    const int tp = (a.L + 15) / 16 * 16;
#define INTEL_TRUNK(TPV)                                                            \
    case TPV:                                                                       \
        return a.heads == 1 ? trunk_launch<TPV, 32>(a, bwd, s) : trunk_launch<TPV, 16>(a, bwd, s);
    switch (tp) {
        INTEL_TRUNK(16) INTEL_TRUNK(32) INTEL_TRUNK(48) INTEL_TRUNK(64)
    }
#undef INTEL_TRUNK
    set_error("fused stack: unsupported padded length %d", tp);
    return INTEL_ERR_UNSUPPORTED;
}

static TrunkArgs trunk_args(int64_t B, int64_t L, int heads, int layers, const StackParams& p, float* const* X,
                            const StackSaved& sv, float drop_p, uint64_t drop_seed, int stream_id) {
    TrunkArgs a;
    memset(&a, 0, sizeof(a));
    for (int l = 0; l < 8; ++l) a.drop[l] = make_dropout(drop_p, drop_seed, stream_id, l);
    for (int l = 0; l < layers && l < 8; ++l) {
        a.QKV[l] = sv.QKV[l]; a.A[l] = sv.A[l]; a.U[l] = sv.U[l]; a.Z[l] = sv.Z[l]; a.ST[l] = sv.ST[l];
    }
    a.save = 1;
    a.B = B; a.L = (int)L; a.heads = heads; a.layers = layers;
    a.wq = p.wq; a.wk = p.wk; a.wv = p.wv; a.w1 = p.w1; a.b1 = p.b1; a.w2 = p.w2; a.b2 = p.b2; a.lnw = p.lnw; a.lnb = p.lnb;
    for (int l = 0; l <= layers && l < 9; ++l) a.X[l] = X[l];
    return a;
}

int trunk_fwd(int64_t B, int64_t L, int heads, int layers, const StackParams& p, float* const* X, const StackSaved& sv,
              float drop_p, uint64_t drop_seed, int stream_id, cudaStream_t s, bool save) {
    TrunkArgs a = trunk_args(B, L, heads, layers, p, X, sv, drop_p, drop_seed, stream_id);
    a.save = save ? 1 : 0;
    return trunk_run(a, false, s);
}

int trunk_bwd(int64_t B, int64_t L, int heads, int layers, const StackParams& p, const StackGrads& g, float* const* X,
              const StackSaved& sv, float* dX, float drop_p, uint64_t drop_seed, int stream_id, cudaStream_t s) {
    TrunkArgs a = trunk_args(B, L, heads, layers, p, X, sv, drop_p, drop_seed, stream_id);
    a.dX = dX;
    a.gwq = g.wq; a.gwk = g.wk; a.gwv = g.wv; a.gw1 = g.w1; a.gb1 = g.b1; a.gw2 = g.w2; a.gb2 = g.b2; a.glnw = g.lnw; a.glnb = g.lnb;
    return trunk_run(a, true, s);
}

}  // namespace intel
