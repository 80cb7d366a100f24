// Fused self-attention stack of IntEL.predict_ensemble (IntEL.py:182-197, layers.py:31-60) on the 5th-generation
// tensor cores: tcgen05.mma with accumulators AND the A operands in tensor memory (TMEM).  Forward pass, stream
// width 32, list length L <= 128; writes exactly the activations trunk_bwd_kernel (trunk.cu) reads back.
//
// Mapping.  A tile is 128 token rows = the 128 TMEM lanes: 4 sessions of <= 32 slots, 2 sessions of <= 64 or one of
// <= 128.  A warpgroup (4 warps) owns a tile and thread t owns token row t for the whole stack: tcgen05.ld / st give
// it its own lane, so softmax, bias, ReLU, residual and LayerNorm are thread-local (no shuffles).  Every product is
// 3xTF32 (a_lo b_hi + a_hi b_lo + a_hi b_hi, fp32 accumulation) like the rest of the library:
//   q|k|v = X [Wq;Wk;Wv]^T   A = X hi/lo planes in TMEM (tcgen05.st by the row owners), B = weight planes in smem, N = 96
//   S_h   = Q_h K_h^T         A = Q hi/lo in TMEM, B = the session's K rows in smem (K-major), N = padded keys;
//                             the sessions of a tile write the SAME accumulator columns under a disable-output-lane mask
//   O_h   = P_h V_h           A = exp(S - max) hi/lo written over S in TMEM, B = the session's V^T (transposing scalar
//                             stores, chunk stride 528 B keeps them conflict-free), rows scaled by 1/sum afterwards
//   U = A W1^T + b1, Z = relu(U) W2^T + b2 (+ dropout, + X), LayerNorm
// Only K and V^T (and the weights) live in shared memory: 65 KB per tile, so two warpgroups = two tiles share an SM and
// one computes while the other waits for its MMAs (tcgen05.commit -> mbarrier).  Lists of 65..128 slots need all 512
// TMEM columns for one tile (scores + probabilities of both heads) and run one warpgroup per CTA.
#include "kernels.h"
#include "mma.cuh"
#ifndef INTEL_EMU
#include "tc05.cuh"

namespace intel {

namespace {

constexpr int TC_WQKV_HI = 0, TC_WQKV_LO = 12288, TC_W1_HI = 24576, TC_W1_LO = 28672, TC_W2_HI = 32768, TC_W2_LO = 36864;
constexpr int TC_VEC = 40960, TC_BAR = 41472, TC_TMEM = 41488, TC_WG = 41600;
constexpr int TC_K_HI = 0, TC_K_LO = 16384, TC_VT_HI = 32768, TC_VT_LO = 49664, TC_WG_BYTES = 66560;
constexpr int TC_K_LBO = 2048;       // K planes [k-chunk][128 rows][4]
constexpr int TC_VT_LBO = 528;       // V^T planes [key-chunk][32 channels][4] + 16 B: transposing stores hit 32 banks

__device__ __forceinline__ void split32(const float (&v)[32], uint32_t (&h)[32], uint32_t (&l)[32]) {
#pragma unroll
    for (int j = 0; j < 32; ++j) split_tf32(v[j], h[j], l[j]);
}

// thread's row of a [*, ld] fp32 tensor -> 32 registers (dead rows read as zero)
__device__ __forceinline__ void load_row(float (&v)[32], const float* __restrict__ src, bool live) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 x = live ? *reinterpret_cast<const float4*>(src + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[4 * j] = x.x; v[4 * j + 1] = x.y; v[4 * j + 2] = x.z; v[4 * j + 3] = x.w;
    }
}
__device__ __forceinline__ void store_row(float* dst, const float (&v)[32], bool live) {
    if (!live) return;
#pragma unroll
    for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(dst + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

// weight W [32][32] (nn.Linear: [out][in]) -> K-major hi / lo planes, plane row = row0 + out of `rows` rows; one 16-byte
// plane unit (4 consecutive in-channels of one out-channel) per thread: a float4 load, two 16-byte stores
__device__ __forceinline__ void stage_weight(uint8_t* hi, uint8_t* lo, const float* __restrict__ W, int rows, int row0) {
    for (int e = threadIdx.x; e < TD * TD / 4; e += blockDim.x) {
        const int kq = e >> 5, n = e & 31;
        const float4 v = *reinterpret_cast<const float4*>(W + n * TD + 4 * kq);
        uint4 h, l;
        split_tf32(v.x, h.x, l.x);
        split_tf32(v.y, h.y, l.y);
        split_tf32(v.z, h.z, l.z);
        split_tf32(v.w, h.w, l.w);
        const int off = (kq * rows + row0 + n) * 16;
        *reinterpret_cast<uint4*>(hi + off) = h;
        *reinterpret_cast<uint4*>(lo + off) = l;
    }
}

// three MMAs of one 8-wide k-slice: D (+)= A B with A in tensor memory
__device__ __forceinline__ void mma3_ts(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint64_t b_hi, uint64_t b_lo, uint32_t idesc, bool first) {
    tc05::mma_ts(d, a_lo, b_hi, idesc, first ? 0u : 1u);
    tc05::mma_ts(d, a_hi, b_lo, idesc, 1u);
    tc05::mma_ts(d, a_hi, b_hi, idesc, 1u);
}
__device__ __forceinline__ void mma3_ts(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint64_t b_hi, uint64_t b_lo, uint32_t idesc, bool first,
                                        const tc05::LaneMask& m) {
    tc05::mma_ts(d, a_lo, b_hi, idesc, first ? 0u : 1u, m);
    tc05::mma_ts(d, a_hi, b_lo, idesc, 1u, m);
    tc05::mma_ts(d, a_hi, b_hi, idesc, 1u, m);
}

}  // namespace

// descriptor of the same layout `bytes` further into shared memory
__device__ __forceinline__ uint64_t desc_at(uint64_t base, uint32_t bytes) { return base + (uint64_t)(bytes >> 4); }

// exp(x) for x <= 0 as one FFMA + MUFU.EX2 (relative error 2^-22, far inside the 1e-5 budget of the softmax)
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// SR: slots of a tile reserved per session (32 / 64 / 128), NCH * 32 = KP: padded key count (>= L),
// COLS: tensor-memory columns of one warpgroup
template <int HEADS, int NCH>
__global__ void __launch_bounds__(256, 1) trunk_tc_fwd_kernel(TrunkArgs a, int COLS) {
    constexpr int DK = TD / HEADS, KP = 32 * NCH;
    constexpr int SR = NCH == 1 ? 32 : (NCH == 2 ? 64 : 128), NS = 128 / SR;
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    uint8_t* sm = tc_smem;
    const int tid = threadIdx.x, g = tid >> 7, t = tid & 127, warp = t >> 5;
    const int WGS = blockDim.x >> 7;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + TC_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + TC_TMEM);
    const float* vec = reinterpret_cast<const float*>(sm + TC_VEC);

    // ---- one-time set-up: weight planes, vectors, barriers, tensor memory ----
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wq, 96, 0);
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wk, 96, 32);
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wv, 96, 64);
    stage_weight(sm + TC_W1_HI, sm + TC_W1_LO, a.w1, 32, 0);
    stage_weight(sm + TC_W2_HI, sm + TC_W2_LO, a.w2, 32, 0);
    if (tid < TD) {
        float* v = reinterpret_cast<float*>(sm + TC_VEC);
        v[tid] = a.b1[tid]; v[TD + tid] = a.b2[tid]; v[2 * TD + tid] = a.lnw[tid]; v[3 * TD + tid] = a.lnb[tid];
    }
    if (tid == 0) {
        tc05::mbar_init(&bars[0], 1);
        tc05::mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 32) tc05::tmem_alloc(tmem_slot, 512);
    tc05::fence_smem_to_mma();
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();

    const uint32_t tm = *tmem_slot + (uint32_t)(g * COLS);         // this warpgroup's columns, lane 0
    const uint32_t tl = tm + ((uint32_t)(warp * 32) << 16);         // ... this warp's 32 lanes
    const uint32_t cA = 0, cS = 64, cPlo = 64 + HEADS * KP, cO = 0;
    uint64_t* bar = &bars[g];
    uint32_t phase = 0;
    uint8_t* wg = sm + TC_WG + g * TC_WG_BYTES;
    const uint32_t s_wqkv_hi = tc05::smem_u32(sm + TC_WQKV_HI), s_wqkv_lo = tc05::smem_u32(sm + TC_WQKV_LO);
    const uint32_t s_w1_hi = tc05::smem_u32(sm + TC_W1_HI), s_w1_lo = tc05::smem_u32(sm + TC_W1_LO);
    const uint32_t s_w2_hi = tc05::smem_u32(sm + TC_W2_HI), s_w2_lo = tc05::smem_u32(sm + TC_W2_LO);
    const uint32_t s_k_hi = tc05::smem_u32(wg + TC_K_HI), s_k_lo = tc05::smem_u32(wg + TC_K_LO);
    const uint32_t s_vt_hi = tc05::smem_u32(wg + TC_VT_HI), s_vt_lo = tc05::smem_u32(wg + TC_VT_LO);
    const uint64_t d_wqkv_hi = tc05::make_desc(s_wqkv_hi, 1536, 128), d_wqkv_lo = tc05::make_desc(s_wqkv_lo, 1536, 128);
    const uint64_t d_w1_hi = tc05::make_desc(s_w1_hi, 512, 128), d_w1_lo = tc05::make_desc(s_w1_lo, 512, 128);
    const uint64_t d_w2_hi = tc05::make_desc(s_w2_hi, 512, 128), d_w2_lo = tc05::make_desc(s_w2_lo, 512, 128);
    const uint64_t d_k_hi = tc05::make_desc(s_k_hi, TC_K_LBO, 128), d_k_lo = tc05::make_desc(s_k_lo, TC_K_LBO, 128);
    const uint64_t d_vt_hi = tc05::make_desc(s_vt_hi, TC_VT_LBO, 128), d_vt_lo = tc05::make_desc(s_vt_lo, TC_VT_LBO, 128);
    const uint32_t id_qkv = tc05::make_idesc(128, 96), id_s = tc05::make_idesc(128, KP), id_pv = tc05::make_idesc(128, DK),
                   id_ffn = tc05::make_idesc(128, 32);
    const int pv_steps = (a.L + 7) >> 3;                             // key slices of 8 that hold a live key

    const int L = a.L;
    const int slot = t / SR, r = t - slot * SR;                     // session slot of the tile, row inside the session
    constexpr int vt_sess = (SR >> 2) * TC_VT_LBO;                  // bytes of one session's V^T plane
    const float sl2 = 1.4426950408889634f / sqrtf((float)DK);       // softmax scale folded into the base-2 exponent
    const int64_t tiles = (a.B + NS - 1) / NS;
    const int bar_id = 1 + g;

    // all row owners are done writing operands -> the elected thread may issue
#define TC_PUBLISH()              \
    do {                          \
        tc05::wait_st();          \
        tc05::fence_smem_to_mma(); \
        tc05::fence_before();     \
        bar_sync(bar_id, 128);    \
    } while (0)
#define TC_WAIT()                     \
    do {                              \
        tc05::mbar_wait(bar, phase);  \
        phase ^= 1u;                  \
        tc05::fence_after();          \
    } while (0)

    for (int64_t tile = (int64_t)blockIdx.x * WGS + g; tile < tiles; tile += (int64_t)gridDim.x * WGS) {
        const int64_t b = tile * NS + slot;
        const bool live = b < a.B && r < L;
        const int64_t grow = b * L + r;                              // token row in the [B*L, *] tensors
        float x[32];
        load_row(x, a.X[0] + grow * TD, live);

        for (int l = 0; l < a.layers; ++l) {
            // ---- q|k|v ----
            {
                uint32_t h[32], lo[32];
                split32(x, h, lo);
                tc05::st32(tl + cA, h);
                tc05::st32(tl + cA + 32, lo);
            }
            TC_PUBLISH();
            if (warp == 0) {
                tc05::fence_after();
                if (tc05::elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3_ts(tm + cS, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_wqkv_hi, ks * 2 * 1536),
                                desc_at(d_wqkv_lo, ks * 2 * 1536), id_qkv, ks == 0);
                    tc05::commit(bar);
                }
                __syncwarp();
            }
            // the layer input goes to HBM while the product runs (layer 0's input is the caller's X[0])
            if (l > 0 && a.save) store_row(a.X[l] + grow * TD, x, live);
            TC_WAIT();
            {
                uint32_t uq[32], uk[32], uv[32], h[32], lo[32];
                tc05::ld32(tl + cS, uq);
                tc05::ld32(tl + cS + 32, uk);
                tc05::ld32(tl + cS + 64, uv);
                tc05::wait_ld();
                // Q -> A operand of the score products
#pragma unroll
                for (int j = 0; j < 32; ++j) split_tf32(__uint_as_float(uq[j]), h[j], lo[j]);
                tc05::st32(tl + cA, h);
                tc05::st32(tl + cA + 32, lo);
                // K -> the tile's key planes (row = tile row; dead rows hold zeros)
#pragma unroll
                for (int j = 0; j < 32; ++j) split_tf32(__uint_as_float(uk[j]), h[j], lo[j]);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    *reinterpret_cast<uint4*>(wg + TC_K_HI + c * TC_K_LBO + t * 16) = make_uint4(h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
                    *reinterpret_cast<uint4*>(wg + TC_K_LO + c * TC_K_LBO + t * 16) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                }
                // V -> the session's V^T planes
#pragma unroll
                for (int j = 0; j < 32; ++j) split_tf32(__uint_as_float(uv[j]), h[j], lo[j]);
                const int vo = slot * vt_sess + (r >> 2) * TC_VT_LBO + (r & 3) * 4;
#pragma unroll
                for (int ch = 0; ch < 32; ++ch) {
                    *reinterpret_cast<uint32_t*>(wg + TC_VT_HI + vo + ch * 16) = h[ch];
                    *reinterpret_cast<uint32_t*>(wg + TC_VT_LO + vo + ch * 16) = lo[ch];
                }
                // ---- scores of every head and session ----
                TC_PUBLISH();
                if (warp == 0) {
                    tc05::fence_after();
                    if (tc05::elect_one()) {
#pragma unroll
                        for (int hd = 0; hd < HEADS; ++hd)
#pragma unroll
                            for (int ss = 0; ss < NS; ++ss) {
                                const tc05::LaneMask m = tc05::mask_rows(ss * SR, SR);
#pragma unroll
                                for (int ks = 0; ks < DK / 8; ++ks) {
                                    const uint32_t koff = (uint32_t)((hd * (DK / 4) + 2 * ks) * TC_K_LBO + ss * SR * 16);
                                    mma3_ts(tm + cS + hd * KP, tm + cA + hd * DK + 8 * ks, tm + cA + 32 + hd * DK + 8 * ks,
                                            desc_at(d_k_hi, koff), desc_at(d_k_lo, koff), id_s, ks == 0, m);
                                }
                            }
                        tc05::commit(bar);
                    }
                    __syncwarp();
                }
                if (a.save && live) {            // q | k | v rows for the backward pass, behind the score products
                    float* dst = a.QKV[l] + grow * 3 * TD;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        *reinterpret_cast<uint4*>(dst + 4 * j) = make_uint4(uq[4 * j], uq[4 * j + 1], uq[4 * j + 2], uq[4 * j + 3]);
                        *reinterpret_cast<uint4*>(dst + TD + 4 * j) = make_uint4(uk[4 * j], uk[4 * j + 1], uk[4 * j + 2], uk[4 * j + 3]);
                        *reinterpret_cast<uint4*>(dst + 2 * TD + 4 * j) = make_uint4(uv[4 * j], uv[4 * j + 1], uv[4 * j + 2], uv[4 * j + 3]);
                    }
                }
            }
            TC_WAIT();
            // ---- softmax numerators over S (in place) and the attention output, head by head ----
            float inv[HEADS];
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                const uint32_t cs = cS + hd * KP;
                float mx = -INFINITY, sum = 0.f;
                if (NCH <= 2) {                                  // the whole row of scores stays in registers
                    uint32_t u[NCH][32], h[32], lo[32];
#pragma unroll
                    for (int c = 0; c < NCH; ++c) tc05::ld32(tl + cs + 32 * c, u[c]);
                    tc05::wait_ld();
#pragma unroll
                    for (int c = 0; c < NCH; ++c)
#pragma unroll
                        for (int j = 0; j < 32; ++j) mx = fmaxf(mx, (32 * c + j < L) ? __uint_as_float(u[c][j]) : -INFINITY);
                    const float sh = -mx * sl2;
                    if (hd > 0) TC_WAIT();                       // the previous head's P V product is done with the shared lo plane
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float e = (32 * c + j < L) ? ex2_approx(fmaf(__uint_as_float(u[c][j]), sl2, sh)) : 0.f;
                            sum += e;
                            split_tf32(e, h[j], lo[j]);
                        }
                        tc05::st32(tl + cs + 32 * c, h);
                        tc05::st32(tl + cPlo + 32 * c, lo);
                    }
                } else {
                    for (int c = 0; c < KP; c += 32) {
                        uint32_t u[32];
                        tc05::ld32(tl + cs + c, u);
                        tc05::wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; ++j) mx = fmaxf(mx, (c + j < L) ? __uint_as_float(u[j]) : -INFINITY);
                    }
                    const float sh = -mx * sl2;
                    if (hd > 0) TC_WAIT();
                    for (int c = 0; c < KP; c += 32) {
                        uint32_t u[32], h[32], lo[32];
                        tc05::ld32(tl + cs + c, u);
                        tc05::wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float e = (c + j < L) ? ex2_approx(fmaf(__uint_as_float(u[j]), sl2, sh)) : 0.f;
                            sum += e;
                            split_tf32(e, h[j], lo[j]);
                        }
                        tc05::st32(tl + cs + c, h);
                        tc05::st32(tl + cPlo + c, lo);
                    }
                }
                inv[hd] = 1.0f / sum;
                TC_PUBLISH();
                if (warp == 0) {
                    tc05::fence_after();
                    if (tc05::elect_one()) {
#pragma unroll
                        for (int ss = 0; ss < NS; ++ss) {
                            const tc05::LaneMask m = tc05::mask_rows(ss * SR, SR);
#pragma unroll 2
                            for (int ks = 0; ks < pv_steps; ++ks) {
                                const uint32_t voff = (uint32_t)(ss * vt_sess + hd * DK * 16 + ks * 2 * TC_VT_LBO);
                                mma3_ts(tm + cO + hd * DK, tm + cs + 8 * ks, tm + cPlo + 8 * ks, desc_at(d_vt_hi, voff), desc_at(d_vt_lo, voff),
                                        id_pv, ks == 0, m);
                            }
                        }
                        tc05::commit(bar);
                    }
                    __syncwarp();
                }
            }
            TC_WAIT();
            // ---- FFN ----
            {
                uint32_t u[32], h[32], lo[32];
                float att[32];
                tc05::ld32(tl + cO, u);
                tc05::wait_ld();
#pragma unroll
                for (int j = 0; j < 32; ++j) att[j] = __uint_as_float(u[j]) * inv[j / DK];
                split32(att, h, lo);
                tc05::st32(tl + cA, h);
                tc05::st32(tl + cA + 32, lo);
                TC_PUBLISH();
                if (warp == 0) {
                    tc05::fence_after();
                    if (tc05::elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            mma3_ts(tm + cS, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_w1_hi, ks * 2 * 512), desc_at(d_w1_lo, ks * 2 * 512),
                                    id_ffn, ks == 0);
                        tc05::commit(bar);
                    }
                    __syncwarp();
                }
                if (a.save) store_row(a.A[l] + grow * TD, att, live);
            }
            TC_WAIT();
            {
                uint32_t u[32], h[32], lo[32];
                float uu[32];
                tc05::ld32(tl + cS, u);
                tc05::wait_ld();
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    uu[j] = __uint_as_float(u[j]) + vec[j];
                    split_tf32(fmaxf(uu[j], 0.f), h[j], lo[j]);
                }
                tc05::st32(tl + cA, h);
                tc05::st32(tl + cA + 32, lo);
                TC_PUBLISH();
                if (warp == 0) {
                    tc05::fence_after();
                    if (tc05::elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            mma3_ts(tm + cS + 32, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_w2_hi, ks * 2 * 512),
                                    desc_at(d_w2_lo, ks * 2 * 512), id_ffn, ks == 0);
                        tc05::commit(bar);
                    }
                    __syncwarp();
                }
                if (a.save) store_row(a.U[l] + grow * TD, uu, live);
            }
            TC_WAIT();
            // ---- Z = dropout(F) + X, LayerNorm (the row is in this thread's registers) ----
            {
                uint32_t u[32];
                float z[32];
                tc05::ld32(tl + cS + 32, u);
                tc05::wait_ld();
                const Dropout& dr = a.drop[l];
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    z[j] = (__uint_as_float(u[j]) + vec[TD + j]) * dropout_scale(dr, grow, j, TD) + x[j];
                    sum += z[j];
                }
                const float mean = sum * (1.0f / TD);
                float var = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float d0 = z[j] - mean;
                    var = fmaf(d0, d0, var);
                }
                const float rstd = rsqrtf(var * (1.0f / TD) + 1e-5f);
#pragma unroll
                for (int j = 0; j < 32; ++j) x[j] = live ? (z[j] - mean) * rstd * vec[2 * TD + j] + vec[3 * TD + j] : 0.f;
                if (a.save) {
                    store_row(a.Z[l] + grow * TD, z, live);
                    if (live) *reinterpret_cast<float2*>(a.ST[l] + grow * 2) = make_float2(mean, rstd);
                }
            }
        }
        store_row(a.X[a.layers] + grow * TD, x, live);
    }
#undef TC_PUBLISH
#undef TC_WAIT
    tc05::fence_before();
    __syncthreads();
    if (tid < 32) tc05::tmem_free(*tmem_slot, 512);
}

// ------------------------------------------------------------------------------------------------
// Lists of 129..208 slots (BASELINE.json configs[3]: 200 candidates): a session spans two 128-row tiles.  One warpgroup
// per CTA; thread t owns rows t and 128 + t.  Per layer: q|k|v of both tiles first (K rows and V^T columns of all keys go
// to shared memory, the Q rows to an fp32 stash), then per tile and head S = Q_h K_h^T over all keys (N = padded key
// count, no lane mask), softmax in 32-column passes over tensor memory, O_h = P V_h, and the FFN + LayerNorm of the tile.
// Tensor memory: A planes 64 | O 32 | S / P hi KP | P lo KP  (KP <= 208 -> 512 columns).  A second warpgroup shares the tile's
// tensor-memory lanes and takes every other 32-column chunk of the two softmax passes.
namespace {
constexpr int TL_K_LBO = 4096;                                  // K planes [k-chunk][256 rows][4]
constexpr int TL_K_HI = 0, TL_K_LO = 32768, TL_VT_HI = 65536, TL_VT_LO = 65536 + 28672, TL_Q = 65536 + 2 * 28672;
constexpr int TL_BYTES = TL_Q + 256 * 128;                       // + Q stash [256 rows][32 floats], 16-byte chunks rotated by row
}  // namespace

template <int HEADS>
__global__ void __launch_bounds__(256, 1) trunk_tc_long_fwd_kernel(TrunkArgs a, int KP) {
    constexpr int DK = TD / HEADS;
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    uint8_t* sm = tc_smem;
    // two warpgroups on the one tile: warpgroup 0 owns the rows (thread t = row t: operands, FFN, LayerNorm, stores);
    // warpgroup 1 shares its tensor-memory lanes (warps w and w + 4 see the same 32 lanes) and takes every other 32-column
    // chunk of the softmax passes, which are three quarters of the thread work at 200 keys
    const int tid = threadIdx.x, g = tid >> 7, t = tid & 127, warp = t >> 5;
    uint64_t* bar = reinterpret_cast<uint64_t*>(sm + TC_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + TC_TMEM);
    const float* vec = reinterpret_cast<const float*>(sm + TC_VEC);
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wq, 96, 0);
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wk, 96, 32);
    stage_weight(sm + TC_WQKV_HI, sm + TC_WQKV_LO, a.wv, 96, 64);
    stage_weight(sm + TC_W1_HI, sm + TC_W1_LO, a.w1, 32, 0);
    stage_weight(sm + TC_W2_HI, sm + TC_W2_LO, a.w2, 32, 0);
    if (tid < TD) {
        float* v = reinterpret_cast<float*>(sm + TC_VEC);
        v[tid] = a.b1[tid]; v[TD + tid] = a.b2[tid]; v[2 * TD + tid] = a.lnw[tid]; v[3 * TD + tid] = a.lnb[tid];
    }
    if (tid == 0) {
        tc05::mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 32) tc05::tmem_alloc(tmem_slot, 512);
    tc05::fence_smem_to_mma();
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    const uint32_t tm = *tmem_slot;
    const uint32_t tl = tm + ((uint32_t)(warp * 32) << 16);
    const uint32_t cA = 0, cO = 64, cS = 96, cPlo = 96 + KP;
    uint32_t phase = 0;
    uint8_t* wg = sm + TC_WG;
    const uint64_t d_wqkv_hi = tc05::make_desc(tc05::smem_u32(sm + TC_WQKV_HI), 1536, 128), d_wqkv_lo = tc05::make_desc(tc05::smem_u32(sm + TC_WQKV_LO), 1536, 128);
    const uint64_t d_w1_hi = tc05::make_desc(tc05::smem_u32(sm + TC_W1_HI), 512, 128), d_w1_lo = tc05::make_desc(tc05::smem_u32(sm + TC_W1_LO), 512, 128);
    const uint64_t d_w2_hi = tc05::make_desc(tc05::smem_u32(sm + TC_W2_HI), 512, 128), d_w2_lo = tc05::make_desc(tc05::smem_u32(sm + TC_W2_LO), 512, 128);
    const uint64_t d_k_hi = tc05::make_desc(tc05::smem_u32(wg + TL_K_HI), TL_K_LBO, 128), d_k_lo = tc05::make_desc(tc05::smem_u32(wg + TL_K_LO), TL_K_LBO, 128);
    const uint64_t d_vt_hi = tc05::make_desc(tc05::smem_u32(wg + TL_VT_HI), TC_VT_LBO, 128), d_vt_lo = tc05::make_desc(tc05::smem_u32(wg + TL_VT_LO), TC_VT_LBO, 128);
    const uint32_t id_qkv = tc05::make_idesc(128, 96), id_s = tc05::make_idesc(128, KP), id_pv = tc05::make_idesc(128, DK),
                   id_ffn = tc05::make_idesc(128, 32);
    const int L = a.L, pv_steps = (L + 7) >> 3;
    const float sl2 = 1.4426950408889634f / sqrtf((float)DK);
    float* qs = reinterpret_cast<float*>(wg + TL_Q);
    float* pstat = reinterpret_cast<float*>(wg + TL_BYTES);          // [2 warpgroups][128 rows]: partial row max / row sum
    const bool rows = g == 0;                                        // this thread owns a tile row

#define TL_PUBLISH()               \
    do {                           \
        tc05::wait_st();           \
        tc05::fence_smem_to_mma(); \
        tc05::fence_before();      \
        __syncthreads();           \
    } while (0)
#define TL_WAIT()                    \
    do {                             \
        tc05::mbar_wait(bar, phase); \
        phase ^= 1u;                 \
        tc05::fence_after();         \
    } while (0)

    for (int64_t b = blockIdx.x; b < a.B; b += gridDim.x) {
        float x[2][32];
        bool live[2];
        int64_t grow[2];
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) {
            const int r = tt * 128 + t;
            live[tt] = rows && r < L;
            grow[tt] = b * L + r;
            load_row(x[tt], a.X[0] + grow[tt] * TD, live[tt]);
        }
        for (int l = 0; l < a.layers; ++l) {
            // ---- q|k|v of both tiles ----
#pragma unroll
            for (int tt = 0; tt < 2; ++tt) {
                const int r = tt * 128 + t;
                if (rows) {
                    uint32_t h[32], lo[32];
                    split32(x[tt], h, lo);
                    tc05::st32(tl + cA, h);
                    tc05::st32(tl + cA + 32, lo);
                }
                TL_PUBLISH();
                if (warp == 0 && rows) {
                    tc05::fence_after();
                    if (tc05::elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            mma3_ts(tm + cS, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_wqkv_hi, ks * 2 * 1536),
                                    desc_at(d_wqkv_lo, ks * 2 * 1536), id_qkv, ks == 0);
                        tc05::commit(bar);
                    }
                    __syncwarp();
                }
                if (l > 0 && a.save) store_row(a.X[l] + grow[tt] * TD, x[tt], live[tt]);
                TL_WAIT();
                if (!rows) continue;                                  // the rest of this step is row-owner work without barriers
                uint32_t uq[32], uk[32], uv[32], h[32], lo[32];
                tc05::ld32(tl + cS, uq);
                tc05::ld32(tl + cS + 32, uk);
                tc05::ld32(tl + cS + 64, uv);
                tc05::wait_ld();
#pragma unroll
                for (int c = 0; c < 8; ++c)          // Q stash: this thread's own row, chunk order rotated against bank conflicts
                    *reinterpret_cast<uint4*>(qs + r * 32 + ((c + t) & 7) * 4) = make_uint4(uq[4 * c], uq[4 * c + 1], uq[4 * c + 2], uq[4 * c + 3]);
#pragma unroll
                for (int j = 0; j < 32; ++j) split_tf32(__uint_as_float(uk[j]), h[j], lo[j]);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    *reinterpret_cast<uint4*>(wg + TL_K_HI + c * TL_K_LBO + r * 16) = make_uint4(h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
                    *reinterpret_cast<uint4*>(wg + TL_K_LO + c * TL_K_LBO + r * 16) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) split_tf32(__uint_as_float(uv[j]), h[j], lo[j]);
                if (r < KP) {                          // key slots beyond the padded count are never read
                    const int vo = (r >> 2) * TC_VT_LBO + (r & 3) * 4;
#pragma unroll
                    for (int ch = 0; ch < 32; ++ch) {
                        *reinterpret_cast<uint32_t*>(wg + TL_VT_HI + vo + ch * 16) = h[ch];
                        *reinterpret_cast<uint32_t*>(wg + TL_VT_LO + vo + ch * 16) = lo[ch];
                    }
                }
                if (a.save && live[tt]) {
                    float* dst = a.QKV[l] + grow[tt] * 3 * TD;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        *reinterpret_cast<uint4*>(dst + 4 * j) = make_uint4(uq[4 * j], uq[4 * j + 1], uq[4 * j + 2], uq[4 * j + 3]);
                        *reinterpret_cast<uint4*>(dst + TD + 4 * j) = make_uint4(uk[4 * j], uk[4 * j + 1], uk[4 * j + 2], uk[4 * j + 3]);
                        *reinterpret_cast<uint4*>(dst + 2 * TD + 4 * j) = make_uint4(uv[4 * j], uv[4 * j + 1], uv[4 * j + 2], uv[4 * j + 3]);
                    }
                }
            }
            // ---- attention + FFN, tile by tile ----
#pragma unroll 1
            for (int tt = 0; tt < 2; ++tt) {
                const int r = tt * 128 + t;
                const bool lv = rows && r < L;
                const int64_t gr = b * L + r;
                float inv[HEADS];
#pragma unroll
                for (int hd = 0; hd < HEADS; ++hd) {
                    if (rows && hd == 0) {
                        uint32_t h[32], lo[32];
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const uint4 q4 = *reinterpret_cast<const uint4*>(qs + r * 32 + ((c + t) & 7) * 4);
                            split_tf32(__uint_as_float(q4.x), h[4 * c], lo[4 * c]);
                            split_tf32(__uint_as_float(q4.y), h[4 * c + 1], lo[4 * c + 1]);
                            split_tf32(__uint_as_float(q4.z), h[4 * c + 2], lo[4 * c + 2]);
                            split_tf32(__uint_as_float(q4.w), h[4 * c + 3], lo[4 * c + 3]);
                        }
                        tc05::st32(tl + cA, h);
                        tc05::st32(tl + cA + 32, lo);
                    }
                    TL_PUBLISH();
                    if (warp == 0 && rows) {
                        tc05::fence_after();
                        if (tc05::elect_one()) {
#pragma unroll
                            for (int ks = 0; ks < DK / 8; ++ks) {
                                const uint32_t koff = (uint32_t)((hd * (DK / 4) + 2 * ks) * TL_K_LBO);
                                mma3_ts(tm + cS, tm + cA + hd * DK + 8 * ks, tm + cA + 32 + hd * DK + 8 * ks, desc_at(d_k_hi, koff),
                                        desc_at(d_k_lo, koff), id_s, ks == 0);
                            }
                            tc05::commit(bar);
                        }
                        __syncwarp();
                    }
                    TL_WAIT();
                    // softmax numerators: warpgroup g takes the 32-column chunks c with (c / 32) % 2 == g
                    float mx = -INFINITY, sum = 0.f;
                    for (int c = 32 * g; c < KP; c += 64) {
                        if (c + 32 <= KP) {
                            uint32_t u[32];
                            tc05::ld32(tl + cS + c, u);
                            tc05::wait_ld();
#pragma unroll
                            for (int j = 0; j < 32; ++j) mx = fmaxf(mx, (c + j < L) ? __uint_as_float(u[j]) : -INFINITY);
                        } else {
                            uint32_t u[16];
                            tc05::ld16(tl + cS + c, u);
                            tc05::wait_ld();
#pragma unroll
                            for (int j = 0; j < 16; ++j) mx = fmaxf(mx, (c + j < L) ? __uint_as_float(u[j]) : -INFINITY);
                        }
                    }
                    pstat[g * 128 + t] = mx;
                    __syncthreads();
                    mx = fmaxf(pstat[t], pstat[128 + t]);
                    __syncthreads();                                  // the slots are reused for the sums below
                    const float sh = -mx * sl2;
                    for (int c = 32 * g; c < KP; c += 64) {
                        if (c + 32 <= KP) {
                            uint32_t u[32], h[32], lo[32];
                            tc05::ld32(tl + cS + c, u);
                            tc05::wait_ld();
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const float e = (c + j < L) ? ex2_approx(fmaf(__uint_as_float(u[j]), sl2, sh)) : 0.f;
                                sum += e;
                                split_tf32(e, h[j], lo[j]);
                            }
                            tc05::st32(tl + cS + c, h);
                            tc05::st32(tl + cPlo + c, lo);
                        } else {
                            uint32_t u[16], h[16], lo[16];
                            tc05::ld16(tl + cS + c, u);
                            tc05::wait_ld();
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const float e = (c + j < L) ? ex2_approx(fmaf(__uint_as_float(u[j]), sl2, sh)) : 0.f;
                                sum += e;
                                split_tf32(e, h[j], lo[j]);
                            }
                            tc05::st16(tl + cS + c, h);
                            tc05::st16(tl + cPlo + c, lo);
                        }
                    }
                    pstat[g * 128 + t] = sum;
                    TL_PUBLISH();
                    inv[hd] = 1.0f / (pstat[t] + pstat[128 + t]);
                    if (warp == 0 && rows) {
                        tc05::fence_after();
                        if (tc05::elect_one()) {
#pragma unroll 2
                            for (int ks = 0; ks < pv_steps; ++ks) {
                                const uint32_t voff = (uint32_t)(hd * DK * 16 + ks * 2 * TC_VT_LBO);
                                mma3_ts(tm + cO + hd * DK, tm + cS + 8 * ks, tm + cPlo + 8 * ks, desc_at(d_vt_hi, voff), desc_at(d_vt_lo, voff),
                                        id_pv, ks == 0);
                            }
                            tc05::commit(bar);
                        }
                        __syncwarp();
                    }
                    TL_WAIT();
                    __syncthreads();                                  // every thread has read the sums: the next head may overwrite them
                }
                // FFN
                {
                    float att[32];
                    if (rows) {
                        uint32_t u[32], h[32], lo[32];
                        tc05::ld32(tl + cO, u);
                        tc05::wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; ++j) att[j] = __uint_as_float(u[j]) * inv[j / DK];
                        split32(att, h, lo);
                        tc05::st32(tl + cA, h);
                        tc05::st32(tl + cA + 32, lo);
                    }
                    TL_PUBLISH();
                    if (warp == 0 && rows) {
                        tc05::fence_after();
                        if (tc05::elect_one()) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                mma3_ts(tm + cS, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_w1_hi, ks * 2 * 512), desc_at(d_w1_lo, ks * 2 * 512),
                                        id_ffn, ks == 0);
                            tc05::commit(bar);
                        }
                        __syncwarp();
                    }
                    if (rows && a.save) store_row(a.A[l] + gr * TD, att, lv);
                }
                TL_WAIT();
                {
                    float uu[32];
                    if (rows) {
                        uint32_t u[32], h[32], lo[32];
                        tc05::ld32(tl + cS, u);
                        tc05::wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            uu[j] = __uint_as_float(u[j]) + vec[j];
                            split_tf32(fmaxf(uu[j], 0.f), h[j], lo[j]);
                        }
                        tc05::st32(tl + cA, h);
                        tc05::st32(tl + cA + 32, lo);
                    }
                    TL_PUBLISH();
                    if (warp == 0 && rows) {
                        tc05::fence_after();
                        if (tc05::elect_one()) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                mma3_ts(tm + cS + 32, tm + cA + 8 * ks, tm + cA + 32 + 8 * ks, desc_at(d_w2_hi, ks * 2 * 512),
                                        desc_at(d_w2_lo, ks * 2 * 512), id_ffn, ks == 0);
                            tc05::commit(bar);
                        }
                        __syncwarp();
                    }
                    if (rows && a.save) store_row(a.U[l] + gr * TD, uu, lv);
                }
                TL_WAIT();
                if (rows) {
                    uint32_t u[32];
                    float z[32];
                    tc05::ld32(tl + cS + 32, u);
                    tc05::wait_ld();
                    const Dropout& dr = a.drop[l];
                    float sum = 0.f;
                    // x[tt] with a run-time tt: both copies are updated under a predicate, so the array stays in registers
                    float xin[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) xin[j] = tt == 0 ? x[0][j] : x[1][j];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        z[j] = (__uint_as_float(u[j]) + vec[TD + j]) * dropout_scale(dr, gr, j, TD) + xin[j];
                        sum += z[j];
                    }
                    const float mean = sum * (1.0f / TD);
                    float var = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float d0 = z[j] - mean;
                        var = fmaf(d0, d0, var);
                    }
                    const float rstd = rsqrtf(var * (1.0f / TD) + 1e-5f);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float y = lv ? (z[j] - mean) * rstd * vec[2 * TD + j] + vec[3 * TD + j] : 0.f;
                        if (tt == 0) x[0][j] = y;
                        else x[1][j] = y;
                    }
                    if (a.save) {
                        store_row(a.Z[l] + gr * TD, z, lv);
                        if (lv) *reinterpret_cast<float2*>(a.ST[l] + gr * 2) = make_float2(mean, rstd);
                    }
                }
            }
        }
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) store_row(a.X[a.layers] + grow[tt] * TD, x[tt], live[tt]);
    }
#undef TL_PUBLISH
#undef TL_WAIT
    tc05::fence_before();
    __syncthreads();
    if (tid < 32) tc05::tmem_free(*tmem_slot, 512);
}

static int g_use_tc = 1;
void trunk_debug_use_tcgen05(int on) { g_use_tc = on ? 1 : 0; }

bool trunk_tc_supported(const TrunkArgs& a) {
    return g_use_tc && a.L >= 1 && a.L <= 208 && (a.heads == 1 || a.heads == 2) && a.layers >= 1 && a.layers <= 8;
}

template <int HEADS, int NCH>
static void trunk_tc_launch(const TrunkArgs& a, int WGS, unsigned grid, size_t smem, cudaStream_t s) {
    auto k = trunk_tc_fwd_kernel<HEADS, NCH>;
    ensure_smem(k, smem);
    LAUNCH(k, dim3(grid), dim3(128 * WGS), smem, s, a, 512 / WGS);
}

int trunk_tc_fwd(const TrunkArgs& a, cudaStream_t s) {
    if (a.L > 128) {                                               // two row tiles per session
        const int KP = (a.L + 15) / 16 * 16;
        const size_t smem = (size_t)TC_WG + TL_BYTES + 2 * 128 * 4;      // + the partial row statistics of the two warpgroups
        const unsigned grid = stream_grid(a.B, 1);
        if (a.heads == 1) {
            auto k = trunk_tc_long_fwd_kernel<1>;
            ensure_smem(k, smem);
            LAUNCH(k, dim3(grid), dim3(256), smem, s, a, KP);
        } else {
            auto k = trunk_tc_long_fwd_kernel<2>;
            ensure_smem(k, smem);
            LAUNCH(k, dim3(grid), dim3(256), smem, s, a, KP);
        }
        const double tok = (double)a.B * a.L;
        return check_launch("trunk_fwd", tok * (4.0 * TD + (a.save ? 4.0 * (3 * TD + 4 * TD + 2) * a.layers : 4.0 * TD)),
                            tok * a.layers * (2.0 * 5 * TD * TD + 4.0 * a.L * TD));
    }
    const int NCH = (a.L + 31) / 32;
    const int SR = NCH == 1 ? 32 : (NCH == 2 ? 64 : 128);
    const int need = 64 + (a.heads + 1) * 32 * NCH;                // A planes | S (P hi) per head | P lo
    const int WGS = need <= 256 ? 2 : 1;
    const size_t smem = (size_t)TC_WG + (size_t)WGS * TC_WG_BYTES;
    const int64_t tiles = ceil_div(a.B, 128 / SR);
    const unsigned grid = stream_grid(ceil_div(tiles, WGS), 1);
#define TC_CASE(H, N) if (a.heads == H && NCH == N) trunk_tc_launch<H, N>(a, WGS, grid, smem, s)
    TC_CASE(1, 1); TC_CASE(1, 2); TC_CASE(1, 3); TC_CASE(1, 4);
    TC_CASE(2, 1); TC_CASE(2, 2); TC_CASE(2, 3); TC_CASE(2, 4);
#undef TC_CASE
    const double tok = (double)a.B * a.L;
    const double flops = tok * a.layers * (2.0 * 5 * TD * TD + 4.0 * a.L * TD);
    const double bytes = tok * (4.0 * TD + (a.save ? 4.0 * (3 * TD + 4 * TD + 2) * a.layers : 4.0 * TD));
    return check_launch("trunk_fwd", bytes, flops);
}

}  // namespace intel
#else   // INTEL_EMU: the emulator has no tensor memory; the mma.sync kernels of trunk.cu cover the same math there
namespace intel {
void trunk_debug_use_tcgen05(int) {}
bool trunk_tc_supported(const TrunkArgs&) { return false; }
int trunk_tc_fwd(const TrunkArgs&, cudaStream_t) { return INTEL_ERR_UNSUPPORTED; }
}  // namespace intel
#endif
