// GRU4RecEncoder recurrence (GeneralSeq.py:58-78 -> torch.nn.GRU, gate order r,z,n) for hidden size 128, the size the
// reference hard-codes (GRU4RecEncoder(hidden_size=128), IntEL.py:105-106).  The input projections W_ih x are one GEMM over
// all live history rows, issued by the caller; the recurrence itself is ONE kernel per direction: a CTA owns a tile of
// sessions for all T steps, W_hh (384x128 fp32 = 192 KB) stays in shared memory for the whole kernel, the hidden
// state of the tile lives in shared memory / registers, gh = W_hh h is formed by 3xTF32 tensor-core MMAs and the gate math
// runs in the MMA epilogue on the accumulator fragments (each warp owns 16 hidden units: its r, z and n columns of a unit
// land in the same lane).  HBM traffic is just gi in, h_all / gates out.  gru_tc.cu has the tcgen05 forward kernel.
// Packed-sequence semantics: a session stops updating once t >= len, so h_all[:, T] is its last state.
#include "kernels.h"
#include "mma.cuh"

namespace intel {

static const int GH = 128;              // hidden size
static const int GW = GH + 4;           // smem row stride of W_hh / h tiles (conflict-free fragment reads)
static const int GF_SB = 32;            // sessions per CTA, forward
static const int GB_SB = 16;            // sessions per CTA, backward
static const int GD = 3 * GH + 4;       // smem row stride of the dgh tile

__device__ __forceinline__ void stage_whh(float* Ws, const float* __restrict__ w_hh) {
    for (int e = threadIdx.x; e < 3 * GH * (GH / 4); e += blockDim.x) {
        const int n = e / (GH / 4), k4 = (e % (GH / 4)) * 4;
        *reinterpret_cast<float4*>(Ws + n * GW + k4) = *reinterpret_cast<const float4*>(w_hh + n * GH + k4);
    }
}

__global__ void __launch_bounds__(256, 1) gru_seq_fwd_kernel(int64_t B, int64_t T, const int64_t* __restrict__ lens,
                                                             const float* __restrict__ gi,
                                                             const float* __restrict__ w_hh,
                                                             const float* __restrict__ b_hh, float* __restrict__ h_all,
                                                             float* __restrict__ gates) {
    DYN_SMEM(float, sm);
    float* Ws = sm;                          // [384][GW]
    float* hs = Ws + 3 * GH * GW;            // [GF_SB][GW]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int64_t b0 = (int64_t)blockIdx.x * GF_SB;
    stage_whh(Ws, w_hh);
    for (int e = threadIdx.x; e < GF_SB * GW; e += blockDim.x) hs[e] = 0.f;
    // rows of this lane: r = i*16 + hh*8 + gq (i: m-tile, hh: half); columns: c = 16*warp + 8*ct + 2*tq + e
    int64_t len_r[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int64_t b = b0 + (q >> 1) * 16 + (q & 1) * 8 + gq;
        len_r[q] = (b < B) ? lens[b] : 0;
    }
    float bias[3][2][2];
#pragma unroll
    for (int gte = 0; gte < 3; ++gte)
#pragma unroll
        for (int ct = 0; ct < 2; ++ct)
#pragma unroll
            for (int e = 0; e < 2; ++e) bias[gte][ct][e] = b_hh[gte * GH + 16 * warp + 8 * ct + 2 * tq + e];
    __syncthreads();

    for (int64_t t = 0; t < T; ++t) {
        // this step's input pre-activations: requested before the recurrent product so that the HBM latency is hidden
        float2 gin[2][2][2][3];             // [m-tile][half][ct][gate]
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int64_t b = b0 + i * 16 + hh * 8 + gq;
                const bool live = (b < B) && (t < len_r[i * 2 + hh]);
#pragma unroll
                for (int ct = 0; ct < 2; ++ct)
#pragma unroll
                    for (int gte = 0; gte < 3; ++gte)
                        gin[i][hh][ct][gte] = live ? *reinterpret_cast<const float2*>(gi + (b * T + t) * 3 * GH + gte * GH + 16 * warp + 8 * ct + 2 * tq)
                                                   : make_float2(0.f, 0.f);
            }
        float acc[2][6][4];                 // [m-tile][gate*2 + ct][frag]
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;
#pragma unroll 2
        for (int ks = 0; ks < GH / 8; ++ks) {
            const int k0 = ks * 8 + tq;
            uint32_t ah[2][4], al[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                split_tf32(hs[(i * 16 + gq) * GW + k0], ah[i][0], al[i][0]);
                split_tf32(hs[(i * 16 + gq + 8) * GW + k0], ah[i][1], al[i][1]);
                split_tf32(hs[(i * 16 + gq) * GW + k0 + 4], ah[i][2], al[i][2]);
                split_tf32(hs[(i * 16 + gq + 8) * GW + k0 + 4], ah[i][3], al[i][3]);
            }
            uint32_t bh[6][2], bl[6][2];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const int n = (j >> 1) * GH + 16 * warp + 8 * (j & 1) + gq;
                split_tf32(Ws[n * GW + k0], bh[j][0], bl[j][0]);
                split_tf32(Ws[n * GW + k0 + 4], bh[j][1], bl[j][1]);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 6; ++j) mma_tf32(acc[i][j], al[i], bh[j]);
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 6; ++j) mma_tf32(acc[i][j], ah[i], bl[j]);
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 6; ++j) mma_tf32(acc[i][j], ah[i], bh[j]);
        }
        // ---- gates on the accumulator fragments ----
        float hn[2][2][2][2];               // [m-tile][half][ct][e]
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int row = i * 16 + hh * 8 + gq;
                const int64_t b = b0 + row;
                const bool live = (b < B) && (t < len_r[i * 2 + hh]);
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) {
                    const int c = 16 * warp + 8 * ct + 2 * tq;
                    const float hp0 = hs[row * GW + c], hp1 = hs[row * GW + c + 1];
                    float o0 = hp0, o1 = hp1;
                    if (live) {
                        const float2 ir = gin[i][hh][ct][0], iz = gin[i][hh][ct][1], in = gin[i][hh][ct][2];
                        const float r0 = sigmoidf_(ir.x + acc[i][0 + ct][2 * hh] + bias[0][ct][0]);
                        const float r1 = sigmoidf_(ir.y + acc[i][0 + ct][2 * hh + 1] + bias[0][ct][1]);
                        const float z0 = sigmoidf_(iz.x + acc[i][2 + ct][2 * hh] + bias[1][ct][0]);
                        const float z1 = sigmoidf_(iz.y + acc[i][2 + ct][2 * hh + 1] + bias[1][ct][1]);
                        const float g0 = acc[i][4 + ct][2 * hh] + bias[2][ct][0];
                        const float g1 = acc[i][4 + ct][2 * hh + 1] + bias[2][ct][1];
                        const float n0 = tanhf(in.x + r0 * g0), n1 = tanhf(in.y + r1 * g1);
                        o0 = (1.f - z0) * n0 + z0 * hp0;
                        o1 = (1.f - z1) * n1 + z1 * hp1;
                        float* gt = gates + (b * T + t) * 4 * GH;
                        *reinterpret_cast<float2*>(gt + c) = make_float2(r0, r1);
                        *reinterpret_cast<float2*>(gt + GH + c) = make_float2(z0, z1);
                        *reinterpret_cast<float2*>(gt + 2 * GH + c) = make_float2(n0, n1);
                        *reinterpret_cast<float2*>(gt + 3 * GH + c) = make_float2(g0, g1);
                    }
                    hn[i][hh][ct][0] = o0;
                    hn[i][hh][ct][1] = o1;
                    if (b < B) *reinterpret_cast<float2*>(h_all + (b * (T + 1) + t + 1) * GH + c) = make_float2(o0, o1);
                }
            }
        __syncthreads();                    // every warp has finished reading the old state
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) {
                    const int row = i * 16 + hh * 8 + gq, c = 16 * warp + 8 * ct + 2 * tq;
                    hs[row * GW + c] = hn[i][hh][ct][0];
                    hs[row * GW + c + 1] = hn[i][hh][ct][1];
                }
        __syncthreads();
    }
}

// h_all[:, 0] must be zero (the caller clears it); h_all [B, T+1, 128], gates [B, T, 512]
int gru_seq_fwd(int64_t B, int64_t T, const int64_t* lens, const float* gi, const float* w_hh, const float* b_hh, float* h_all,
                float* gates, cudaStream_t s) {
    if (B <= 0 || T <= 0) return INTEL_OK;
    const size_t smem = (size_t)(3 * GH * GW + GF_SB * GW) * 4;
    ensure_smem(gru_seq_fwd_kernel, smem);
    LAUNCH(gru_seq_fwd_kernel, dim3((unsigned)ceil_div(B, GF_SB)), dim3(256), smem, s, B, T, lens, gi, w_hh, b_hh, h_all,
           gates);
    return check_launch("gru_seq_fwd", (double)B * T * (3 + 4 + 1) * GH * 4.0, 2.0 * B * T * 3 * GH * GH);
}

// ------------------------------------------------------------------------------------------------
// Output projections of the two GRU encoders (GeneralSeq.py:76-77: out = Linear(128 -> d, no bias) of the last state) and
// their input gradients, both encoders in one launch: a [4096 x 48..64 x 128] product is far too small for a GEMM launch of
// its own (four launches of 22 us each in round 2).  One warp per session; W [n][128] sits in shared memory with row stride 129.
namespace {
constexpr int OP_H = 128, OP_WS = OP_H + 1, OP_WARPS = 8, OP_NMAX = 64;
struct OutProjArgs {
    int64_t B;
    int n[2];
    const float* W[2];
    const float* x[2]; int64_t ldx[2];      // forward: the last states; backward: d(out) rows
    float* y[2]; int64_t ldy[2];            // forward: out rows; backward: d(last state) [B, 128]
};
}  // namespace

__global__ void __launch_bounds__(OP_WARPS * 32) gru_outproj_fwd_kernel(OutProjArgs a) {
    DYN_SMEM(float, sm);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* Ws[2] = {sm, sm + OP_NMAX * OP_WS};
    float* xb = sm + 2 * OP_NMAX * OP_WS + w * OP_H;
    // weights -> shared memory with independent 16-byte loads (nn.Linear weights are 16-byte aligned allocations)
    for (int i = 0; i < 2; ++i) {
#pragma unroll 8
        for (int e = threadIdx.x; e < a.n[i] * (OP_H / 4); e += blockDim.x) {
            const float4 v = *reinterpret_cast<const float4*>(a.W[i] + 4 * e);
            float* dst = Ws[i] + (e >> 5) * OP_WS + 4 * (e & 31);
            dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
        }
    }
    __syncthreads();
    const int64_t nwarps = (int64_t)gridDim.x * OP_WARPS;
    for (int64_t b = (int64_t)blockIdx.x * OP_WARPS + w; b < a.B; b += nwarps) {
        for (int i = 0; i < 2; ++i) {
            const float4 v = *reinterpret_cast<const float4*>(a.x[i] + b * a.ldx[i] + 4 * lane);
            __syncwarp();
            *reinterpret_cast<float4*>(xb + 4 * lane) = v;
            __syncwarp();
            const int j0 = lane, j1 = lane + 32;
            const bool on0 = j0 < a.n[i], on1 = j1 < a.n[i];
            const float* w0 = Ws[i] + (on0 ? j0 : 0) * OP_WS;
            const float* w1 = Ws[i] + (on1 ? j1 : 0) * OP_WS;
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll 8
            for (int u = 0; u < OP_H; u += 4) {
                const float4 h4 = *reinterpret_cast<const float4*>(xb + u);
                acc0 = fmaf(h4.x, w0[u], fmaf(h4.y, w0[u + 1], fmaf(h4.z, w0[u + 2], fmaf(h4.w, w0[u + 3], acc0))));
                acc1 = fmaf(h4.x, w1[u], fmaf(h4.y, w1[u + 1], fmaf(h4.z, w1[u + 2], fmaf(h4.w, w1[u + 3], acc1))));
            }
            if (on0) a.y[i][b * a.ldy[i] + j0] = acc0;
            if (on1) a.y[i][b * a.ldy[i] + j1] = acc1;
        }
    }
}

// d(last state)[b, u] = sum_j d(out)[b, j] W[j][u]
__global__ void __launch_bounds__(OP_WARPS * 32) gru_outproj_dx_kernel(OutProjArgs a) {
    DYN_SMEM(float, sm);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* Ws[2] = {sm, sm + OP_NMAX * OP_WS};
    float* gb = sm + 2 * OP_NMAX * OP_WS + w * OP_NMAX;
    // weights -> shared memory with independent 16-byte loads (nn.Linear weights are 16-byte aligned allocations)
    for (int i = 0; i < 2; ++i) {
#pragma unroll 8
        for (int e = threadIdx.x; e < a.n[i] * (OP_H / 4); e += blockDim.x) {
            const float4 v = *reinterpret_cast<const float4*>(a.W[i] + 4 * e);
            float* dst = Ws[i] + (e >> 5) * OP_WS + 4 * (e & 31);
            dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
        }
    }
    __syncthreads();
    const int64_t nwarps = (int64_t)gridDim.x * OP_WARPS;
    for (int64_t b = (int64_t)blockIdx.x * OP_WARPS + w; b < a.B; b += nwarps) {
        for (int i = 0; i < 2; ++i) {
            __syncwarp();
            gb[lane] = lane < a.n[i] ? a.x[i][b * a.ldx[i] + lane] : 0.f;
            gb[lane + 32] = lane + 32 < a.n[i] ? a.x[i][b * a.ldx[i] + lane + 32] : 0.f;
            __syncwarp();
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int j = 0; j < a.n[i]; ++j) {
                const float g = gb[j];
                const float* wr = Ws[i] + j * OP_WS + lane;
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[q] = fmaf(g, wr[32 * q], acc[q]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) a.y[i][b * a.ldy[i] + lane + 32 * q] = acc[q];
        }
    }
}

bool gru_outproj_pair_ok(int n0, int n1) { return n0 >= 1 && n0 <= OP_NMAX && n1 >= 1 && n1 <= OP_NMAX; }

static int gru_outproj_launch(bool dx, int64_t B, const int* n, const float* const* W, const float* const* x, const int64_t* ldx,
                              float* const* y, const int64_t* ldy, cudaStream_t s) {
    if (B <= 0) return INTEL_OK;
    OutProjArgs a;
    a.B = B;
    for (int i = 0; i < 2; ++i) {
        a.n[i] = n[i]; a.W[i] = W[i]; a.x[i] = x[i]; a.ldx[i] = ldx[i]; a.y[i] = y[i]; a.ldy[i] = ldy[i];
        INTEL_REQUIRE(dx || (ldx[i] % 4 == 0 && (uintptr_t)x[i] % 16 == 0), INTEL_ERR_ARG, "gru_outproj: state rows must be 16-byte aligned");
        INTEL_REQUIRE((uintptr_t)W[i] % 16 == 0, INTEL_ERR_ARG, "gru_outproj: weights must be 16-byte aligned");
    }
    const size_t smem = (size_t)(2 * OP_NMAX * OP_WS + OP_WARPS * OP_H) * 4;
    const unsigned grid = stream_grid(ceil_div(B, OP_WARPS), 2);
    if (dx) {
        ensure_smem(gru_outproj_dx_kernel, smem);
        LAUNCH(gru_outproj_dx_kernel, dim3(grid), dim3(OP_WARPS * 32), smem, s, a);
    } else {
        ensure_smem(gru_outproj_fwd_kernel, smem);
        LAUNCH(gru_outproj_fwd_kernel, dim3(grid), dim3(OP_WARPS * 32), smem, s, a);
    }
    return check_launch(dx ? "gru_outproj_dx" : "gru_outproj_fwd", (double)B * 4.0 * (2 * OP_H + n[0] + n[1]), 2.0 * B * OP_H * (n[0] + n[1]));
}
int gru_outproj_pair_fwd(int64_t B, const int* n, const float* const* W, const float* const* h_last, const int64_t* ldh,
                         float* const* out, const int64_t* ldo, cudaStream_t s) {
    return gru_outproj_launch(false, B, n, W, h_last, ldh, out, ldo, s);
}
int gru_outproj_pair_dx(int64_t B, const int* n, const float* const* W, const float* const* dout, const int64_t* ldd,
                        float* const* dh, const int64_t* ldh, cudaStream_t s) {
    return gru_outproj_launch(true, B, n, W, dout, ldd, dh, ldh, s);
}

// Row numbers of the live (session, step) pairs of a padded [B, T] history, in (b, t) order.  Block k owns sessions
// [1024 k, 1024 k + 1024): it sums the lengths before them, scans its own and writes its rows; the last block writes the count.
__device__ void gru_live_rows_body(int blk, int nblk, int64_t B, int T, const int64_t* __restrict__ lens, int32_t* __restrict__ rows_t,
                                   int32_t* __restrict__ rows_t1, int32_t* __restrict__ count) {
    __shared__ int warp_tot[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto len_of = [&](int64_t e) { const int64_t v = lens[e]; return (int)(v < 0 ? 0 : (v > T ? T : v)); };
    const int64_t first = (int64_t)blk * 1024;
    // lengths before this block
    int part = 0;
    for (int64_t e = tid; e < first; e += 1024) part += len_of(e);
    part = warp_sum_i(part);
    if (lane == 0) warp_tot[warp] = part;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int w = 0; w < 32; ++w) t += warp_tot[w];
        base_s = t;
    }
    __syncthreads();
    const int base = base_s;
    __syncthreads();
    // exclusive scan of the block's own lengths
    const int64_t b = first + tid;
    const int n = b < B ? len_of(b) : 0;
    int incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    const int off = base + before + incl - n;
    // a warp writes the rows of its 32 sessions one session at a time: lane t takes step t (contiguous stores)
    for (int i = 0; i < 32; ++i) {
        const int o = __shfl_sync(0xffffffffu, off, i), m = __shfl_sync(0xffffffffu, n, i);
        const int64_t bb = first + warp * 32 + i;
        for (int t = lane; t < m; t += 32) {
            rows_t[o + t] = (int32_t)(bb * T + t);
            rows_t1[o + t] = (int32_t)(bb * (T + 1) + t);
        }
    }
    if (blk == nblk - 1 && tid == 1023) *count = off + n;
}
// Sessions in order of decreasing length (stable), the way pack_padded_sequence orders them (GeneralSeq.py:64-71): a tile
// of consecutive sessions of that order then shares one loop bound, and tiles that end early make room for the next ones.
// One block; a chunk of 1024 sessions per pass, rank inside a chunk from warp ballots, so the order is deterministic.
__device__ void gru_order_body(int64_t B, int T, const int64_t* __restrict__ lens, int32_t* __restrict__ order) {
    __shared__ int cnt[64], start[64], run[64], wcnt[32][64];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 64) { cnt[tid] = 0; run[tid] = 0; }
    if (tid == 0) order[B] = 0;              // tile counter of the backward recurrence, kept behind the B entries
    __syncthreads();
    auto key = [&](int64_t e) { const int64_t v = lens[e]; return (int)(v < 0 ? 0 : (v > T ? T : v)); };
    for (int64_t c0 = 0; c0 < B; c0 += 1024) {           // histogram: one shared-memory atomic per warp and length
        const int64_t e = c0 + tid;
        const int v = e < B ? key(e) : -1;
        for (int u = 0; u <= T; ++u) {
            const unsigned m = __ballot_sync(0xffffffffu, v == u);
            if (lane == 0 && m) atomicAdd(&cnt[u], __popc(m));
        }
    }
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int v = T; v >= 0; --v) { start[v] = acc; acc += cnt[v]; }
    }
    __syncthreads();
    for (int64_t c0 = 0; c0 < B; c0 += 1024) {
        const int64_t e = c0 + tid;
        const int v = e < B ? key(e) : -1;
        int rank = 0;
        for (int u = 0; u <= T; ++u) {
            const unsigned m = __ballot_sync(0xffffffffu, v == u);
            if (lane == 0) wcnt[warp][u] = __popc(m);
            if (v == u) rank = __popc(m & ((1u << lane) - 1u));
        }
        __syncthreads();
        if (v >= 0) {
            int pre = 0;
            for (int w = 0; w < warp; ++w) pre += wcnt[w][v];
            order[start[v] + run[v] + pre + rank] = (int32_t)e;
        }
        __syncthreads();
        if (tid <= T) {
            int tot = 0;
            for (int w = 0; w < 32; ++w) tot += wcnt[w][tid];
            run[tid] += tot;
        }
        __syncthreads();
    }
}
// One launch prepares both encoders: blocks [0, nb) of row y list the live rows of encoder y, block nb sorts its sessions.
struct GruPrepArgs {
    GruPrepOne e[2];
    int n;
};
__global__ void __launch_bounds__(1024) gru_prep_kernel(GruPrepArgs a) {
    const GruPrepOne& E = a.e[blockIdx.y];
    const int nb = (int)((E.B + 1023) / 1024);
    if ((int)blockIdx.x < nb) {
        if (E.rows_t) gru_live_rows_body((int)blockIdx.x, nb, E.B, E.T, E.lens, E.rows_t, E.rows_t1, E.count);
    } else if ((int)blockIdx.x == nb) {
        if (E.order) gru_order_body(E.B, E.T, E.lens, E.order);
    }
}
int gru_prep(int n, const GruPrepOne* e, cudaStream_t s) {
    GruPrepArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n;
    int64_t nb = 0;
    for (int i = 0; i < n; ++i) {
        INTEL_REQUIRE(e[i].B * (e[i].T + 1) < (1LL << 31) || !e[i].rows_t, INTEL_ERR_UNSUPPORTED, "gru_prep: more than 2^31 history rows");
        INTEL_REQUIRE(!e[i].order || (e[i].T >= 1 && e[i].T <= 63), INTEL_ERR_UNSUPPORTED, "gru_prep: sorting needs T in [1, 63]");
        a.e[i] = e[i];
        const int64_t x = ceil_div(e[i].B, 1024);
        nb = x > nb ? x : nb;
    }
    if (n <= 0 || nb <= 0) return INTEL_OK;
    LAUNCH(gru_prep_kernel, dim3((unsigned)(nb + 1), (unsigned)n), dim3(1024), 0, s, a);
    return check_launch("gru_prep");
}

// Backward recurrence of up to two encoders in one launch (GruBwdOne / GruBwdPair, kernels.h).  dh_in [B,128] holds
// d(loss)/d h_T on entry.  Writes dgi [B,T,384] and dgh_all [B,T+1,384] (slot T untouched) for the weight-gradient GEMMs.
// Each encoder has its own W_hh, and restaging it costs a CTA as much as a few steps: so every CTA draws the tiles of its
// home encoder (blockIdx.x % n) from that encoder's counter, longest first, and only when they are gone the remaining
// (shortest) tiles of the other one.  One launch then balances the SMs over the tiles of both encoders, and no CTA
// stages W_hh more than twice.
__global__ void __launch_bounds__(256, 1) gru_seq_bwd_kernel(GruBwdPair a) {
    DYN_SMEM(float, sm);
    __shared__ int s_tile, s_enc;
    __shared__ float s_bias[2][4][GH];       // per encoder: column sums of dgi (r, z, n) and of the n part of dgh
    float* Ws = sm;                          // [384][GW]   W_hh[k = gate column][n = hidden]
    float* ds = Ws + 3 * GH * GW;            // [GB_SB][GD] dgh of the current step
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    for (int e = threadIdx.x; e < 2 * 4 * GH; e += blockDim.x) (&s_bias[0][0][0])[e] = 0.f;
    const int home = (int)(blockIdx.x % a.n);
    const int64_t ntiles0 = (a.e[0].B + GB_SB - 1) / GB_SB, ntiles1 = a.n > 1 ? (a.e[1].B + GB_SB - 1) / GB_SB : 0;
    int staged = -1;                         // the encoder whose W_hh is in shared memory
    for (int64_t it = 0;; ++it) {
    // next tile: with the length-sorted orders the tiles are handed out longest first from the counters (the CTAs that
    // drew short tiles come back for more), otherwise round robin (one encoder)
    int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
    int enc = 0;
    if (a.e[0].counter) {
        if (threadIdx.x == 0) {
            int e = staged < 0 ? home : staged;
            int t = atomicAdd(e ? a.e[1].counter : a.e[0].counter, 1);
            if (t >= (e ? ntiles1 : ntiles0) && e == home && a.n > 1) {
                e ^= 1;
                t = atomicAdd(e ? a.e[1].counter : a.e[0].counter, 1);
            }
            s_tile = t;
            s_enc = e;
        }
        __syncthreads();
        tile = s_tile;
        enc = s_enc;
    }
    if (tile >= (enc ? ntiles1 : ntiles0)) break;
    const GruBwdOne E = enc ? a.e[1] : a.e[0];
    const int64_t B = E.B, T = E.T;
    const int64_t b0 = tile * GB_SB;
    if (enc != staged) {
        __syncthreads();                     // no warp still reads the other encoder's W_hh
        stage_whh(Ws, E.w_hh);
        staged = enc;
    }
    // the tile's sessions: consecutive entries of the length-sorted order (longest first), so the first one bounds the loop;
    // session slots beyond B are marked with B (every access below is guarded by b < B)
    auto sess = [&](int64_t i) -> int64_t { return i < B ? (E.order ? (int64_t)E.order[i] : i) : B; };
    int64_t tmax = T;
    if (E.order) {
        const int64_t l0 = E.lens[sess(b0)];
        tmax = l0 < 0 ? 0 : (l0 > T ? T : l0);
    }
    // without live_only, gradient rows behind the tile's last live step are zero (a product reads every row)
    if (!E.live_only && tmax < T) {
        const int64_t per = (T - tmax) * (3 * GH / 4);
        for (int64_t e = threadIdx.x; e < (int64_t)GB_SB * per; e += blockDim.x) {
            const int64_t b = sess(b0 + e / per), r = e % per;
            if (b < B) {
                const int64_t t = tmax + r / (3 * GH / 4), c4 = (r % (3 * GH / 4)) * 4;
                *reinterpret_cast<float4*>(E.dgi + (b * T + t) * 3 * GH + c4) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(E.dgh_all + (b * (T + 1) + t) * 3 * GH + c4) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    }
    float sum_i[2][3][2], sum_h[2][2];        // the tile's bias-gradient partial sums: [ct][gate][e] of dgi, [ct][e] of dgh_n
#pragma unroll
    for (int ct = 0; ct < 2; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            sum_h[ct][e] = 0.f;
#pragma unroll
            for (int q = 0; q < 3; ++q) sum_i[ct][q][e] = 0.f;
        }
    int64_t len_r[2], b_r[2];
    float dh[2][2][2];                       // [half][ct][e]: rows gq / gq+8, cols 16*warp + 8*ct + 2*tq + e
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const int64_t b = sess(b0 + hh * 8 + gq);
        b_r[hh] = b;
        len_r[hh] = (b < B) ? E.lens[b] : 0;
#pragma unroll
        for (int ct = 0; ct < 2; ++ct) {
            const int c = 16 * warp + 8 * ct + 2 * tq;
            float2 v = make_float2(0.f, 0.f);
            if (b < B) v = *reinterpret_cast<const float2*>(E.dh_in + b * GH + c);
            dh[hh][ct][0] = v.x;
            dh[hh][ct][1] = v.y;
        }
    }
    __syncthreads();
    // saved gate values r | z | n | W_hn h + b_hn and the previous state of one step, for the elements this lane owns;
    // the values of step t - 1 are requested before the recurrent product of step t (latency hidden behind the MMAs)
    float2 sv[2][2][5];
    auto fetch = [&](int64_t t, float2 (&v)[2][2][5]) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int64_t b = b_r[hh];
            const bool live = (b < B) && (t >= 0) && (t < len_r[hh]);
#pragma unroll
            for (int ct = 0; ct < 2; ++ct) {
                const int c = 16 * warp + 8 * ct + 2 * tq;
#pragma unroll
                for (int q = 0; q < 5; ++q) v[hh][ct][q] = make_float2(0.f, 0.f);
                if (live) {
                    const float* gt = E.gates + (b * T + t) * 4 * GH;
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[hh][ct][q] = *reinterpret_cast<const float2*>(gt + q * GH + c);
                    v[hh][ct][4] = *reinterpret_cast<const float2*>(E.h_all + (b * (T + 1) + t) * GH + c);
                }
            }
        }
    };
    fetch(tmax - 1, sv);
    for (int64_t t = tmax - 1; t >= 0; --t) {
        // ---- gate derivatives for the elements this lane owns ----
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int row = hh * 8 + gq;
            const int64_t b = b_r[hh];
            const bool live = (b < B) && (t < len_r[hh]);
#pragma unroll
            for (int ct = 0; ct < 2; ++ct) {
                const int c = 16 * warp + 8 * ct + 2 * tq;
                float2 dr = make_float2(0.f, 0.f), dz = dr, dn = dr, dnr = dr;
                if (live) {
                    const float2 r = sv[hh][ct][0], z = sv[hh][ct][1], n = sv[hh][ct][2], gn = sv[hh][ct][3], hp = sv[hh][ct][4];
                    const float g0 = dh[hh][ct][0], g1 = dh[hh][ct][1];
                    dn.x = g0 * (1.f - z.x) * (1.f - n.x * n.x);
                    dn.y = g1 * (1.f - z.y) * (1.f - n.y * n.y);
                    dz.x = g0 * (hp.x - n.x) * z.x * (1.f - z.x);
                    dz.y = g1 * (hp.y - n.y) * z.y * (1.f - z.y);
                    dr.x = dn.x * gn.x * r.x * (1.f - r.x);
                    dr.y = dn.y * gn.y * r.y * (1.f - r.y);
                    dnr.x = dn.x * r.x;
                    dnr.y = dn.y * r.y;
                    dh[hh][ct][0] = g0 * z.x;
                    dh[hh][ct][1] = g1 * z.y;
                }
                if (live || (!E.live_only && b < B)) {
                    float* di = E.dgi + (b * T + t) * 3 * GH;
                    float* dg = E.dgh_all + (b * (T + 1) + t) * 3 * GH;
                    *reinterpret_cast<float2*>(di + c) = dr;
                    *reinterpret_cast<float2*>(di + GH + c) = dz;
                    *reinterpret_cast<float2*>(di + 2 * GH + c) = dn;
                    *reinterpret_cast<float2*>(dg + c) = dr;
                    *reinterpret_cast<float2*>(dg + GH + c) = dz;
                    *reinterpret_cast<float2*>(dg + 2 * GH + c) = dnr;
                }
                sum_i[ct][0][0] += dr.x; sum_i[ct][0][1] += dr.y;
                sum_i[ct][1][0] += dz.x; sum_i[ct][1][1] += dz.y;
                sum_i[ct][2][0] += dn.x; sum_i[ct][2][1] += dn.y;
                sum_h[ct][0] += dnr.x;   sum_h[ct][1] += dnr.y;
                ds[row * GD + c] = dr.x;            ds[row * GD + c + 1] = dr.y;
                ds[row * GD + GH + c] = dz.x;       ds[row * GD + GH + c + 1] = dz.y;
                ds[row * GD + 2 * GH + c] = dnr.x;  ds[row * GD + 2 * GH + c + 1] = dnr.y;
            }
        }
        __syncthreads();
        float2 nx[2][2][5];
        fetch(t - 1, nx);
        // ---- dh_prev = dh * z + dgh W_hh : [16 x 384] x [384 x 128], this warp owns 16 output columns ----
        // hi*hi and the two small products go to separate accumulators, and so do even and odd k-slices: eight
        // independent chains of at most 48 dependent MMAs per warp instead of two of 144
        float hi[2][2][4], lo[2][2][4];      // [k-slice parity][ct][frag]
#pragma unroll
        for (int p = 0; p < 2; ++p)
#pragma unroll
            for (int ct = 0; ct < 2; ++ct)
#pragma unroll
                for (int c = 0; c < 4; ++c) hi[p][ct][c] = lo[p][ct][c] = 0.f;
#pragma unroll 2
        for (int ks = 0; ks < 3 * GH / 8; ks += 2) {
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                const int k0 = (ks + p) * 8 + tq;
                uint32_t ah[4], al[4];
                split_tf32(ds[gq * GD + k0], ah[0], al[0]);
                split_tf32(ds[(gq + 8) * GD + k0], ah[1], al[1]);
                split_tf32(ds[gq * GD + k0 + 4], ah[2], al[2]);
                split_tf32(ds[(gq + 8) * GD + k0 + 4], ah[3], al[3]);
                uint32_t bh[2][2], bl[2][2];
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) {
                    const int n = 16 * warp + 8 * ct + gq;
                    split_tf32(Ws[k0 * GW + n], bh[ct][0], bl[ct][0]);
                    split_tf32(Ws[(k0 + 4) * GW + n], bh[ct][1], bl[ct][1]);
                }
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) mma_tf32(lo[p][ct], al, bh[ct]);
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) mma_tf32(lo[p][ct], ah, bl[ct]);
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) mma_tf32(hi[p][ct], ah, bh[ct]);
            }
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int ct = 0; ct < 2; ++ct) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int f = 2 * hh + e;
                    dh[hh][ct][e] += (lo[0][ct][f] + lo[1][ct][f]) + (hi[0][ct][f] + hi[1][ct][f]);
                }
#pragma unroll
                for (int q = 0; q < 5; ++q) sv[hh][ct][q] = nx[hh][ct][q];
            }
        __syncthreads();                    // the dgh tile is rewritten by the next step
    }
    // ---- the tile's bias-gradient sums, added to the CTA's per-encoder sums (one owner lane per column) ----
#pragma unroll
    for (int ct = 0; ct < 2; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            float v[4] = {sum_i[ct][0][e], sum_i[ct][1][e], sum_i[ct][2][e], sum_h[ct][e]};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                v[q] += __shfl_xor_sync(0xffffffffu, v[q], 4);
                v[q] += __shfl_xor_sync(0xffffffffu, v[q], 8);
                v[q] += __shfl_xor_sync(0xffffffffu, v[q], 16);
            }
            if (gq == 0) {
                const int c = 16 * warp + 8 * ct + 2 * tq + e;
#pragma unroll
                for (int q = 0; q < 4; ++q) s_bias[enc][q][c] += v[q];
            }
        }
    }   // tile loop
    // ---- bias gradients: db_ih = column sums of dgi, db_hh = column sums of dgh (r and z parts are shared) ----
    __syncthreads();
    for (int i = 0; i < a.n; ++i) {
        float *db_ih = a.e[i].db_ih, *db_hh = a.e[i].db_hh;
        for (int c = threadIdx.x; c < GH; c += blockDim.x) {
            const float r = s_bias[i][0][c], z = s_bias[i][1][c];
            if (db_ih) { atomicAdd(db_ih + c, r); atomicAdd(db_ih + GH + c, z); atomicAdd(db_ih + 2 * GH + c, s_bias[i][2][c]); }
            if (db_hh) { atomicAdd(db_hh + c, r); atomicAdd(db_hh + GH + c, z); atomicAdd(db_hh + 2 * GH + c, s_bias[i][3][c]); }
        }
    }
}

int gru_seq_bwd_pair(const GruBwdPair& p, cudaStream_t s) {
    int64_t tiles = 0;
    double bytes = 0.0, flops = 0.0;
    INTEL_REQUIRE(p.n == 1 || (p.n == 2 && p.e[0].counter && p.e[1].counter), INTEL_ERR_ARG,
                  "gru_seq_bwd: two encoders need a tile counter each");
    for (int i = 0; i < p.n; ++i) {
        const GruBwdOne& o = p.e[i];
        INTEL_REQUIRE(o.B >= 0 && o.T >= 0, INTEL_ERR_ARG, "gru_seq_bwd: bad shape");
        tiles += ceil_div(o.B, GB_SB);
        bytes += (double)o.B * o.T * (4 + 1 + 3 + 3) * GH * 4.0;
        flops += 2.0 * o.B * o.T * 3 * GH * GH;
    }
    if (tiles <= 0) return INTEL_OK;
    const size_t smem = (size_t)(3 * GH * GW + GB_SB * GD) * 4;
    ensure_smem(gru_seq_bwd_kernel, smem);
    // persistent: one CTA per SM (W_hh fills its shared memory)
    LAUNCH(gru_seq_bwd_kernel, dim3(stream_grid(tiles, 1)), dim3(256), smem, s, p);
    return check_launch("gru_seq_bwd", bytes, flops);
}

}  // namespace intel
