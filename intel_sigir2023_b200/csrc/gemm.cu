// Tensor-core GEMM for the dense contractions of the IntEL path (nn.Linear forward, input gradients,
// weight gradients).  fp32 parity (1e-5) rules out plain TF32/BF16 math (SURVEY.md section 7), so every
// product is formed as three m16n8k8 TF32 MMAs on hi/lo splits of the fp32 operands (mma.cuh); the first
// FFMA version of this kernel was instruction-issue bound at 32 % FMA-pipe utilisation
// (profiles/r01_summary.md) - the MMA form issues ~5x fewer instructions per MAC.
//
// All shapes here have a tiny inner dimension (32..384, 1071 at most) or a tiny output, so tiles are
// 128 x {32,64} x 32 with register-staged prefetch of the next k-tile; operands may be stored k-major or
// row-major (the three nn.Linear passes), selected at compile time.
#include <stdarg.h>

#include "kernels.h"
#include "mma.cuh"

namespace intel {

struct GemmDev {
    int64_t M, N, K;
    const float* A; int64_t lda;
    const float* B; int64_t ldb;
    float* C; int64_t ldc;
    const float* bias;
    const float* add; int64_t ldadd;
    const float* mask; int64_t ldmask;
    int relu_a, relu_b, relu_out, accumulate, splits, vec_a, vec_b, vec_c;
    int64_t kchunk;
};

static const int BK = 32;     // k depth of a gemm_tc_kernel stage

// Global -> register staging of one operand tile.  TR = operand stored [K][rows] (rows contiguous),
// otherwise [rows][K] (k contiguous).  Two modes: 16-byte chunks when the operand is 16-byte aligned with a
// leading dimension that is a multiple of 4, otherwise element-wise with consecutive lanes on consecutive
// addresses (I = 1071 makes every operand with that leading dimension misaligned; a per-thread 4-float
// fallback there cost 4x the transactions).  BK: k depth of the tile.
template <int ROWS, int NT, bool TR, int BK>
struct TileLoader {
    static constexpr int CH = ROWS * BK / 4;                 // float4 chunks per tile
    static constexpr int NV = (CH + NT - 1) / NT;
    static constexpr int NE = 4 * NV;                        // scalars per thread
    static constexpr int LD = TR ? ROWS + 8 : BK + 4;       // shared-memory leading dimension
    float f[NE];

    __device__ __forceinline__ void load(const float* __restrict__ P, int64_t ld, int64_t r0, int64_t rmax, int64_t k0,
                                         int64_t kend, int vec, int relu, int tid) {
        if (vec) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int e = tid + i * NT;
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (e < CH) {
                    if (TR) {
                        const int kk = e / (ROWS / 4), r4 = (e % (ROWS / 4)) * 4;
                        const int64_t gk = k0 + kk, gr = r0 + r4;
                        if (gk < kend) {
                            const float* p = P + gk * ld + gr;
                            if (gr + 3 < rmax) x = *reinterpret_cast<const float4*>(p);
                            else {
                                if (gr < rmax) x.x = p[0];
                                if (gr + 1 < rmax) x.y = p[1];
                                if (gr + 2 < rmax) x.z = p[2];
                            }
                        }
                    } else {
                        const int rr = e / (BK / 4), k4 = (e % (BK / 4)) * 4;
                        const int64_t gr = r0 + rr, gk = k0 + k4;
                        if (gr < rmax) {
                            const float* p = P + gr * ld + gk;
                            if (gk + 3 < kend) x = *reinterpret_cast<const float4*>(p);
                            else {
                                if (gk < kend) x.x = p[0];
                                if (gk + 1 < kend) x.y = p[1];
                                if (gk + 2 < kend) x.z = p[2];
                            }
                        }
                    }
                }
                f[4 * i] = x.x; f[4 * i + 1] = x.y; f[4 * i + 2] = x.z; f[4 * i + 3] = x.w;
            }
        } else {
#pragma unroll
            for (int i = 0; i < NE; ++i) {
                const int e = tid + i * NT;
                float x = 0.f;
                if (e < ROWS * BK) {
                    if (TR) {
                        const int kk = e / ROWS, r = e % ROWS;
                        if (k0 + kk < kend && r0 + r < rmax) x = P[(k0 + kk) * ld + r0 + r];
                    } else {
                        const int rr = e / BK, k = e % BK;
                        if (r0 + rr < rmax && k0 + k < kend) x = P[(r0 + rr) * ld + k0 + k];
                    }
                }
                f[i] = x;
            }
        }
        if (relu) {
#pragma unroll
            for (int i = 0; i < NE; ++i) f[i] = fmaxf(f[i], 0.f);
        }
    }
    __device__ __forceinline__ void store(float* s, int vec, int tid) const {
        if (vec) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int e = tid + i * NT;
                if (e < CH) {
                    const float4 x = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
                    if (TR) {
                        const int kk = e / (ROWS / 4), r4 = (e % (ROWS / 4)) * 4;
                        *reinterpret_cast<float4*>(s + kk * LD + r4) = x;
                    } else {
                        const int rr = e / (BK / 4), k4 = (e % (BK / 4)) * 4;
                        *reinterpret_cast<float4*>(s + rr * LD + k4) = x;
                    }
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < NE; ++i) {
                const int e = tid + i * NT;
                if (e < ROWS * BK) {
                    if (TR) s[(e / ROWS) * LD + (e % ROWS)] = f[i];
                    else s[(e / BK) * LD + (e % BK)] = f[i];
                }
            }
        }
    }
};

// element (row r, k) of a staged tile
template <bool TR, int LD>
__device__ __forceinline__ float tile_at(const float* s, int r, int k) { return TR ? s[k * LD + r] : s[r * LD + k]; }

__device__ __forceinline__ void gemm_store(const GemmDev& g, int64_t gm, int64_t gn, float v, bool first) {
    if (gm >= g.M || gn >= g.N) return;
    if (first) {
        if (g.bias) v += g.bias[gn];
        if (g.add) v += g.add[gm * g.ldadd + gn];
    }
    if (g.relu_out) v = fmaxf(v, 0.f);
    if (g.mask) v = (g.mask[gm * g.ldmask + gn] > 0.f) ? v : 0.f;
    float* c = g.C + gm * g.ldc + gn;
    if (g.accumulate == 0) *c = v;
    else if (g.accumulate == 1) *c += v;
    else atomicAdd(c, v);
}

// two adjacent columns (gn even): one 8-byte access per operand when the layout allows it (g.vec_c)
__device__ __forceinline__ void gemm_store2(const GemmDev& g, int64_t gm, int64_t gn, float v0, float v1, bool first) {
    if (gm >= g.M) return;
    if (!g.vec_c || gn + 1 >= g.N) {
        gemm_store(g, gm, gn, v0, first);
        gemm_store(g, gm, gn + 1, v1, first);
        return;
    }
    if (first) {
        if (g.bias) { const float2 b = *reinterpret_cast<const float2*>(g.bias + gn); v0 += b.x; v1 += b.y; }
        if (g.add) { const float2 a = *reinterpret_cast<const float2*>(g.add + gm * g.ldadd + gn); v0 += a.x; v1 += a.y; }
    }
    if (g.relu_out) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
    if (g.mask) {
        const float2 m = *reinterpret_cast<const float2*>(g.mask + gm * g.ldmask + gn);
        v0 = m.x > 0.f ? v0 : 0.f;
        v1 = m.y > 0.f ? v1 : 0.f;
    }
    float* c = g.C + gm * g.ldc + gn;
    if (g.accumulate == 0) *reinterpret_cast<float2*>(c) = make_float2(v0, v1);
    else if (g.accumulate == 1) { float2 o = *reinterpret_cast<float2*>(c); *reinterpret_cast<float2*>(c) = make_float2(o.x + v0, o.y + v1); }
    else { atomicAdd(c, v0); atomicAdd(c + 1, v1); }
}

}  // namespace intel
#include "gemm_umma.cuh"
namespace intel {

template <int BM, int BN, int WM, int WN, bool AT, bool BT>
__global__ void __launch_bounds__(WM * WN * 32) gemm_tc_kernel(GemmDev g) {
    constexpr int NT = WM * WN * 32;
    constexpr int TM = BM / WM / 16, TN = BN / WN / 8;
    using LA = TileLoader<BM, NT, AT, BK>;
    using LB = TileLoader<BN, NT, BT, BK>;
    constexpr int SA = LA::LD, SB = LB::LD;
    __shared__ __align__(16) float sA[AT ? BK * SA : BM * SA];
    __shared__ __align__(16) float sB[BT ? BK * SB : BN * SB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / WN, wn = warp % WN;
    const int gq = lane >> 2, tq = lane & 3;
    const int64_t m0 = (int64_t)blockIdx.x * BM, n0 = (int64_t)blockIdx.y * BN;
    const int64_t kbeg = (int64_t)blockIdx.z * g.kchunk;
    const int64_t kend = (kbeg + g.kchunk < g.K) ? kbeg + g.kchunk : g.K;

    float acc[TM][TN][4];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;

    LA la;
    LB lb;
    if (kbeg < kend) {
        la.load(g.A, g.lda, m0, g.M, kbeg, kend, g.vec_a, g.relu_a, tid);
        lb.load(g.B, g.ldb, n0, g.N, kbeg, kend, g.vec_b, g.relu_b, tid);
    }
    for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
        la.store(sA, g.vec_a, tid);
        lb.store(sB, g.vec_b, tid);
        __syncthreads();
        if (k0 + BK < kend) {     // prefetch the next k-tile into registers while this one is consumed
            la.load(g.A, g.lda, m0, g.M, k0 + BK, kend, g.vec_a, g.relu_a, tid);
            lb.load(g.B, g.ldb, n0, g.N, k0 + BK, kend, g.vec_b, g.relu_b, tid);
        }
        // The tensor core adds into its accumulator with truncation, so a long MMA chain drifts towards zero
        // linearly in K.  Each k-tile is therefore summed from zero in `part` and folded into `acc` with a
        // round-to-nearest FADD.
        float part[TM][TN][4];
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) part[i][j][c] = 0.f;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            const int kb = ks * 8;
            float af[TM][4], bf[TN][2];
#pragma unroll
            for (int i = 0; i < TM; ++i) {
                const int r = wm * (BM / WM) + i * 16 + gq;
                af[i][0] = tile_at<AT, SA>(sA, r, kb + tq);
                af[i][1] = tile_at<AT, SA>(sA, r + 8, kb + tq);
                af[i][2] = tile_at<AT, SA>(sA, r, kb + tq + 4);
                af[i][3] = tile_at<AT, SA>(sA, r + 8, kb + tq + 4);
            }
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                const int c = wn * (BN / WN) + j * 8 + gq;
                bf[j][0] = tile_at<BT, SB>(sB, c, kb + tq);
                bf[j][1] = tile_at<BT, SB>(sB, c, kb + tq + 4);
            }
            uint32_t ah[TM][4], al[TM][4], bh[TN][2], bl[TN][2];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    split_tf32(af[i][c], ah[i][c], al[i][c]);
                }
#pragma unroll
            for (int j = 0; j < TN; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    split_tf32(bf[j][c], bh[j][c], bl[j][c]);
                }
            // three passes over independent accumulators: no back-to-back dependent MMAs
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) mma_tf32(part[i][j], al[i], bh[j]);
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) mma_tf32(part[i][j], ah[i], bl[j]);
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) mma_tf32(part[i][j], ah[i], bh[j]);
        }
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[i][j][c] += part[i][j][c];
        __syncthreads();
    }

    const bool first = (blockIdx.z == 0);
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int64_t gm = m0 + wm * (BM / WM) + i * 16 + gq;
            const int64_t gn = n0 + wn * (BN / WN) + j * 8 + 2 * tq;
            gemm_store2(g, gm, gn, acc[i][j][0], acc[i][j][1], first);
            gemm_store2(g, gm + 8, gn, acc[i][j][2], acc[i][j][3], first);
        }
}

// Split-warp 32 x 32 kernel for products whose output fills too few 128-row tiles while the inner dimension is long:
// tall outputs with few columns (the intent-side projections [B x 1071] x [1071 -> 32]: a 128 x 32 tiling leaves 32-64 CTAs
// walking 34 k-tiles one after the other; A [M][K], B [N][K] or, BT, [K][N]) and weight gradients with a small output
// (AT = BT = true, split-K over blockIdx.z, atomicAdd epilogue).  The eight warps of a CTA take 16 k each of every staged
// 128-deep slab; their partial tiles are summed through shared memory.
static const int SW_BK = 128;
template <bool AT, bool BT>
__global__ void __launch_bounds__(256) gemm_warpsplit_kernel(GemmDev g) {
    using LA = TileLoader<32, 256, AT, SW_BK>;
    using LB = TileLoader<32, 256, BT, SW_BK>;
    constexpr int SA = LA::LD, SB = LB::LD;
    constexpr int NA = AT ? SW_BK * SA : 32 * SA, NB = BT ? SW_BK * SB : 32 * SB;
    __shared__ __align__(16) float sm[NA + NB > 8 * 1024 ? NA + NB : 8 * 1024];     // A slab | B slab, then the 8 partial tiles
    float* sA = sm;
    float* sB = sm + NA;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int64_t m0 = (int64_t)blockIdx.x * 32, n0 = (int64_t)blockIdx.y * 32;
    const int64_t kbeg = (int64_t)blockIdx.z * g.kchunk;
    const int64_t kend = (kbeg + g.kchunk < g.K) ? kbeg + g.kchunk : g.K;
    float acc[2][4][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;

    LA la;
    LB lb;
    if (kbeg < kend) {
        la.load(g.A, g.lda, m0, g.M, kbeg, kend, g.vec_a, g.relu_a, tid);
        lb.load(g.B, g.ldb, n0, g.N, kbeg, kend, g.vec_b, g.relu_b, tid);
    }
    for (int64_t k0 = kbeg; k0 < kend; k0 += SW_BK) {
        la.store(sA, g.vec_a, tid);
        lb.store(sB, g.vec_b, tid);
        __syncthreads();
        if (k0 + SW_BK < kend) {     // next slab in flight while this one is consumed
            la.load(g.A, g.lda, m0, g.M, k0 + SW_BK, kend, g.vec_a, g.relu_a, tid);
            lb.load(g.B, g.ldb, n0, g.N, k0 + SW_BK, kend, g.vec_b, g.relu_b, tid);
        }
        float part[2][4][4];     // per-slab partial sums, folded into acc with a rounded add (see gemm_tc_kernel)
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) part[i][j][c] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int kb = warp * 16 + ks * 8;
            float af[2][4], bf[4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int r = i * 16 + gq;
                af[i][0] = tile_at<AT, SA>(sA, r, kb + tq);
                af[i][1] = tile_at<AT, SA>(sA, r + 8, kb + tq);
                af[i][2] = tile_at<AT, SA>(sA, r, kb + tq + 4);
                af[i][3] = tile_at<AT, SA>(sA, r + 8, kb + tq + 4);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = j * 8 + gq;
                bf[j][0] = tile_at<BT, SB>(sB, c, kb + tq);
                bf[j][1] = tile_at<BT, SB>(sB, c, kb + tq + 4);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) mma_3xtf32(part[i][j], af[i], bf[j]);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[i][j][c] += part[i][j][c];
        __syncthreads();
    }
    float* red = sm + warp * 1024;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = i * 16 + gq, c = j * 8 + 2 * tq;
            red[r * 32 + c] = acc[i][j][0];
            red[r * 32 + c + 1] = acc[i][j][1];
            red[(r + 8) * 32 + c] = acc[i][j][2];
            red[(r + 8) * 32 + c + 1] = acc[i][j][3];
        }
    __syncthreads();
    const bool first = (blockIdx.z == 0);
    for (int e = tid; e < 1024; e += 256) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += sm[w * 1024 + e];
        gemm_store(g, m0 + (e >> 5), n0 + (e & 31), v, first);
    }
}

// Streaming form for the dominant shape of the two self-attention stacks: a very tall A[M,32] against a
// 32 x N (N <= 32) weight.  No shared memory and no barriers: every warp keeps the whole weight as pre-split
// hi/lo B fragments in registers and walks over 16-row m-tiles, reading its A fragments straight from global
// memory.  The MMA k index is a free permutation as long as A and B agree, so k-step s / slot t is mapped to
// memory column 8t + 2s (+1 for the t+4 slot): a lane's eight fragment values of a row are then one
// contiguous 32-byte run (two 16-byte loads), and the four lanes of a row cover its 128 bytes exactly.
template <bool BT>
__global__ void __launch_bounds__(256) gemm_stream32_kernel(GemmDev g) {
    const int lane = threadIdx.x & 31;
    const int gq = lane >> 2, tq = lane & 3;
    const int ntiles = (int)((g.N + 7) / 8);
    uint32_t bh[4][4][2], bl[4][4][2];      // [n-tile][k-step][slot]
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int64_t n = j * 8 + gq;
                const int k = 8 * tq + 2 * s + c;
                float w = 0.f;
                if (j < ntiles && n < g.N) w = BT ? g.B[k * g.ldb + n] : g.B[n * g.ldb + k];
                if (g.relu_b) w = fmaxf(w, 0.f);
                split_tf32(w, bh[j][s][c], bl[j][s][c]);
            }
        }
    }
    const int64_t n_mt = (g.M + 15) / 16;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float4 cur[4], nxt[4];
    auto fetch = [&](int64_t mt, float4 (&v)[4]) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t r = mt * 16 + gq + 8 * h;
            if (r < g.M) {
                const float4* p = reinterpret_cast<const float4*>(g.A + r * g.lda + 8 * tq);
                v[2 * h] = p[0];
                v[2 * h + 1] = p[1];
            } else {
                v[2 * h] = make_float4(0.f, 0.f, 0.f, 0.f);
                v[2 * h + 1] = v[2 * h];
            }
        }
    };
    if (warp0 < n_mt) fetch(warp0, cur);
    for (int64_t mt = warp0; mt < n_mt; mt += nwarps) {
        if (mt + nwarps < n_mt) fetch(mt + nwarps, nxt);
        // this lane's values: row gq -> lo[0..7], row gq+8 -> hi[0..7] (memory columns 8 tq .. 8 tq + 7)
        float lo[8] = {cur[0].x, cur[0].y, cur[0].z, cur[0].w, cur[1].x, cur[1].y, cur[1].z, cur[1].w};
        float hi[8] = {cur[2].x, cur[2].y, cur[2].z, cur[2].w, cur[3].x, cur[3].y, cur[3].z, cur[3].w};
        if (g.relu_a) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { lo[i] = fmaxf(lo[i], 0.f); hi[i] = fmaxf(hi[i], 0.f); }
        }
        float acc[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const float af[4] = {lo[2 * s], hi[2 * s], lo[2 * s + 1], hi[2 * s + 1]};
            uint32_t ah[4], al[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                split_tf32(af[c], ah[c], al[c]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < ntiles) {
                    mma_tf32(acc[j], al, bh[j][s]);
                    mma_tf32(acc[j], ah, bl[j][s]);
                    mma_tf32(acc[j], ah, bh[j][s]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < ntiles) {
                const int64_t gn = j * 8 + 2 * tq;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int64_t gm = mt * 16 + gq + 8 * h;
                    gemm_store2(g, gm, gn, acc[j][2 * h], acc[j][2 * h + 1], true);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) cur[i] = nxt[i];
    }
}

// How gemm() computes one product.  gemm_plan() makes every choice; the launch below follows it.
struct GemmPlan {
    enum Kernel { UMMA, WARPSPLIT, STREAM32, TC } kernel;
    bool prezero;              // C is cleared first and the split partial products are added with atomics
    int splits;                // CTAs along the inner dimension (blockIdx.z), kchunk deep each
    int64_t kchunk;
    int cfg;                   // mma.sync kernels: 0: 128x64  1: 128x32  2: 64x64  3: 64x32  (TC tiles)  4: 32x32 weight gradient
    int bn, nraw, vec_c4;      // UMMA: N tile, raw fp32 stages, 16-byte aligned rows of C / add / mask / bias
    bool multi;                // UMMA: the k range spans several accumulation chunks
    size_t smem;               // UMMA: dynamic shared memory
};

static int g_tcgen05 = 1, g_rows_gemm = 1;
void gemm_debug_use_tcgen05(int on) { g_tcgen05 = on ? 1 : 0; }
void gemm_debug_use_rows_gemm(int on) { g_rows_gemm = on ? 1 : 0; }

static inline bool vec_ok(const float* p, int64_t ld) { return (((uintptr_t)p) % 16 == 0) && (ld % 4 == 0); }

// splits of the inner dimension: enough CTAs for `waves` waves of the SMs, no split shallower than 4 granules; kchunk is a
// multiple of the granule
static void split_k(GemmPlan& p, int64_t K, int64_t tiles, int waves, int granule, bool can_split) {
    int64_t n = 1;
    if (can_split) {
        const int64_t want = ceil_div(waves * kNumSMs, tiles), maxs = ceil_div(K, 4 * granule);
        n = want < maxs ? want : maxs;
        if (n < 1) n = 1;
    }
    p.splits = (int)n;
    p.kchunk = ceil_div(ceil_div(K, n), granule) * granule;
    if (p.kchunk <= 0) p.kchunk = granule;
}

static GemmPlan gemm_plan(const Gemm& g) {
    GemmPlan p{};
    const bool wgrad = g.pass == GemmPass::WGRAD;
    auto ctas = [&](int bm, int bn) { return ceil_div(g.M, bm) * ceil_div(g.N, bn); };
    // plain outputs with a long inner dimension and too few tiles to fill the GPU are split like the weight gradients: the
    // output is cleared first and the partial products are accumulated with atomics
    p.prezero = g.accumulate == 0 && !g.relu_out && !g.mask && g.K >= 512 && g.N > 64 && ctas(128, 64) < kNumSMs;
    const bool can_split = wgrad || p.prezero;
    // tall outputs with few columns and a long inner dimension fill too few 128-row tiles: the warp-split kernel
    const bool skinny = !wgrad && !p.prezero && g.N <= 64 && g.K >= 256 && ctas(128, 32) < 2 * kNumSMs;
#ifndef INTEL_EMU
    // large products: tcgen05 kernel (gemm_umma.cuh), 128 x bn tiles, TMEM accumulators
    if (g_tcgen05 && !skinny && g.M >= 128 && g.N >= 16 && g.K >= 16 && (double)g.M * g.N * g.K >= 134217728.0) {
        p.kernel = GemmPlan::UMMA;
        p.bn = (int)(g.N >= 128 ? 128 : ceil_div(g.N, 16) * 16);
        split_k(p, g.K, ceil_div(g.M, umma::UM) * ceil_div(g.N, p.bn), 3, umma::UBK, can_split);
        // short inner dimension: the epilogue dominates; a 2-deep raw ring keeps two CTAs per SM
        // (up to 256 inner columns the forward layout keeps the 2-deep ring as well - 121 registers, two CTAs per SM: 54 -> 39 us
        // for the pred_layer product; the transposing variants need 154+ registers, one CTA per SM either way)
        p.nraw = (p.kchunk <= 128 || (p.kchunk <= 256 && g.pass == GemmPass::FWD)) ? 2 : 4;
        p.multi = p.kchunk > (int64_t)umma::UCH * umma::UBK;
        p.smem = (size_t)umma::USTAGES * 2 * (umma::plane_bytes(umma::UM) + umma::plane_bytes(p.bn)) +
                 (size_t)p.nraw * (umma::raw_bytes(umma::UM) + umma::raw_bytes(p.bn));
        const size_t tile_bytes = (size_t)umma::UM * (p.bn + 4) * 4;      // epilogue staging tile reuses the operand stages
        if (p.smem < tile_bytes) p.smem = tile_bytes;
        auto al16 = [](const float* q, int64_t ld) { return q == nullptr || vec_ok(q, ld); };
        p.vec_c4 = al16(g.C, g.ldc) && al16(g.add, g.ldadd) && al16(g.mask, g.ldmask) && al16(g.bias, 4);
        return p;
    }
#endif
    // mma.sync kernels: the largest tile that still yields ~2 waves of CTAs on the SMs; weight gradients with a small output
    // take the warp-split kernel
    if (wgrad && (g.M < 64 || g.N < 64)) p.cfg = 4;
    else if (g.N <= 32) p.cfg = (ctas(128, 32) >= 2 * kNumSMs || can_split) ? 1 : 3;
    else if (ctas(128, 64) >= 2 * kNumSMs || can_split) p.cfg = 0;
    else if (ctas(64, 64) >= 2 * kNumSMs) p.cfg = 2;
    else p.cfg = 3;
    const int bm = p.cfg == 4 ? 32 : (p.cfg <= 1 ? 128 : 64), bn = (p.cfg == 0 || p.cfg == 2) ? 64 : 32;
    split_k(p, g.K, ctas(bm, bn), 2, p.cfg == 4 ? SW_BK : BK, can_split);
    if (skinny || p.cfg == 4) p.kernel = GemmPlan::WARPSPLIT;
    else if (!wgrad && g.K == 32 && g.N <= 32 && vec_ok(g.A, g.lda) && g.accumulate != 2 && g.M >= 2048) p.kernel = GemmPlan::STREAM32;
    else p.kernel = GemmPlan::TC;
    return p;
}

template <int BM, int BN, int WM, int WN, bool AT, bool BT>
static void launch_tc(const GemmDev& d, cudaStream_t s) {
    auto k = gemm_tc_kernel<BM, BN, WM, WN, AT, BT>;
    LAUNCH(k, dim3((unsigned)ceil_div(d.M, BM), (unsigned)ceil_div(d.N, BN), (unsigned)d.splits), dim3(WM * WN * 32), 0, s, d);
}

// AT / BT: the operand layouts of the pass
template <bool AT, bool BT>
static void gemm_launch(const GemmDev& d, const GemmPlan& p, cudaStream_t s) {
    switch (p.kernel) {
#ifndef INTEL_EMU
    case GemmPlan::UMMA: {
        using K = void (*)(GemmDev, int, int);
        // [NACC = 32, 64, 128][one accumulation chunk; several chunks with 2 / 4 raw stages]
        static const K kernels[3][3] = {
            {umma::gemm_umma_kernel<AT, BT, 32, false, 2>, umma::gemm_umma_kernel<AT, BT, 32, true, 2>, umma::gemm_umma_kernel<AT, BT, 32, true, 4>},
            {umma::gemm_umma_kernel<AT, BT, 64, false, 2>, umma::gemm_umma_kernel<AT, BT, 64, true, 2>, umma::gemm_umma_kernel<AT, BT, 64, true, 4>},
            {umma::gemm_umma_kernel<AT, BT, 128, false, 2>, umma::gemm_umma_kernel<AT, BT, 128, true, 2>, umma::gemm_umma_kernel<AT, BT, 128, true, 4>}};
        const K k = kernels[p.bn <= 32 ? 0 : (p.bn <= 64 ? 1 : 2)][!p.multi ? 0 : (p.nraw == 2 ? 1 : 2)];
        ensure_smem(k, p.smem);
        const dim3 grid((unsigned)ceil_div(d.M, umma::UM), (unsigned)ceil_div(d.N, p.bn), (unsigned)d.splits);
        LAUNCH(k, grid, dim3(umma::UTHREADS), p.smem, s, d, p.bn, p.vec_c4);
        break;
    }
#endif
    case GemmPlan::WARPSPLIT: {
        auto k = gemm_warpsplit_kernel<AT, BT>;
        LAUNCH(k, dim3((unsigned)ceil_div(d.M, 32), (unsigned)ceil_div(d.N, 32), (unsigned)d.splits), dim3(256), 0, s, d);
        break;
    }
    case GemmPlan::STREAM32: {
        auto k = gemm_stream32_kernel<BT>;
        LAUNCH(k, dim3(stream_grid(ceil_div(d.M, 16 * 8), 3)), dim3(256), 0, s, d);
        break;
    }
    default:
        if (p.cfg == 0) launch_tc<128, 64, 4, 2, AT, BT>(d, s);
        else if (p.cfg == 1) launch_tc<128, 32, 4, 1, AT, BT>(d, s);
        else if (p.cfg == 2) launch_tc<64, 64, 2, 2, AT, BT>(d, s);
        else launch_tc<64, 32, 2, 1, AT, BT>(d, s);
    }
}

int gemm_check_launch(const Gemm& g, const char* tag_fmt, ...) {
    static const char* const names[] = {"gemm_fwd", "gemm_dgrad", "gemm_wgrad"};
    const char* what = names[(int)g.pass];
    if (prof_detail()) {
        char tag[64], name[160];
        va_list ap;
        va_start(ap, tag_fmt);
        vsnprintf(tag, sizeof(tag), tag_fmt, ap);
        va_end(ap);
        snprintf(name, sizeof(name), "%s[%lldx%lldx%lld,%s]", what, (long long)g.M, (long long)g.N, (long long)g.K, tag);
        what = prof_intern(name);
    }
    const double bytes = 4.0 * ((double)g.M * g.K + (double)g.N * g.K +
                                (double)g.M * g.N * (1 + (g.add != nullptr) + (g.mask != nullptr)));
    return check_launch(what, bytes, 2.0 * g.M * g.N * g.K);
}

int gemm(const Gemm& g, cudaStream_t s) {
    if (g.M <= 0 || g.N <= 0) return INTEL_OK;
    INTEL_REQUIRE(g.A && g.B && g.C, INTEL_ERR_ARG, "gemm: null operand");
    INTEL_REQUIRE(g.M <= 0x7fffffffLL * 32 && g.N < (65535LL * 32), INTEL_ERR_ARG, "gemm: shape too large");
    const GemmPlan p = gemm_plan(g);
#ifndef INTEL_EMU
    // tall products with a small resident weight operand, and weight gradients over tens of thousands of rows: the persistent
    // warp-specialised tcgen05 kernels (gemm_rows_tc.cu, gemm_wgrad_tc.cu), when the shape fits them
    if (g_tcgen05 && g_rows_gemm && !p.prezero) {
        int st = 0;
        if (gemm_rows_tc_try(g, s, &st) || gemm_wgrad_tc_try(g, s, &st)) return st;
    }
#endif
    GemmDev d;
    d.M = g.M; d.N = g.N; d.K = g.K;
    d.A = g.A; d.lda = g.lda; d.B = g.B; d.ldb = g.ldb; d.C = g.C; d.ldc = g.ldc;
    d.bias = g.bias; d.add = g.add; d.ldadd = g.ldadd; d.mask = g.mask; d.ldmask = g.ldmask;
    d.relu_a = g.relu_a; d.relu_b = g.relu_b; d.relu_out = g.relu_out; d.accumulate = g.accumulate;
    d.vec_a = vec_ok(g.A, g.lda);
    d.vec_b = vec_ok(g.B, g.ldb);
    auto even = [](const float* q, int64_t ld) { return q == nullptr || ((((uintptr_t)q) % 8 == 0) && (ld % 2 == 0)); };
    d.vec_c = even(g.C, g.ldc) && even(g.add, g.ldadd) && even(g.mask, g.ldmask) && even(g.bias, 2);
    d.splits = p.splits;
    d.kchunk = p.kchunk;
    if (p.prezero) {
        cudaError_t e = cudaMemset2DAsync(g.C, (size_t)g.ldc * 4, 0, (size_t)g.N * 4, (size_t)g.M, s);
        INTEL_REQUIRE(e == cudaSuccess, INTEL_ERR_CUDA, "cudaMemset2DAsync: %s", cudaGetErrorString(e));
        d.accumulate = 2;
    }
    switch (g.pass) {
    case GemmPass::FWD: gemm_launch<false, false>(d, p, s); break;
    case GemmPass::DGRAD: gemm_launch<false, true>(d, p, s); break;
    case GemmPass::WGRAD: gemm_launch<true, true>(d, p, s); break;
    }
    if (p.kernel == GemmPlan::UMMA) return gemm_check_launch(g, "umma,bn%d,splits%d", p.bn, p.splits);
    return gemm_check_launch(g, "cfg%d,splits%d,vec%d%d%d", p.cfg, p.splits, d.vec_a, d.vec_b, d.vec_c);
}

int linear(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const float* W, int64_t ldw,
           const float* bias, float* C, int64_t ldc, cudaStream_t s, bool relu_a, bool relu_out,
           const float* add, int64_t ldadd, const int32_t* rows, const int32_t* nrows) {
    Gemm g;
    g.pass = GemmPass::FWD;
    g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = W; g.ldb = ldw; g.C = C; g.ldc = ldc;
    g.bias = bias; g.relu_a = relu_a; g.relu_out = relu_out; g.add = add; g.ldadd = ldadd; g.rows = rows; g.nrows = nrows;
    return gemm(g, s);
}

bool gemm_rows_only(const Gemm& g) {
#ifndef INTEL_EMU
    if (g.rows && g.nrows && g_tcgen05 && g_rows_gemm && !gemm_plan(g).prezero)
        return gemm_rows_tc_try(g, nullptr, nullptr) || gemm_wgrad_tc_try(g, nullptr, nullptr);
#endif
    return false;
}

Gemm dgrad_gemm(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* W, int64_t ldw, float* dX,
                int64_t lddx, const int32_t* rows, const int32_t* nrows) {
    Gemm g;   // dX[M,K] = dY[M,N] * W[N,K]: inner dimension N, B operand stored [inner][out]
    g.pass = GemmPass::DGRAD;
    g.rows = rows; g.nrows = nrows;
    g.M = M; g.N = K; g.K = N; g.A = dY; g.lda = lddy; g.B = W; g.ldb = ldw;
    g.C = dX; g.ldc = lddx;
    return g;
}

Gemm wgrad_gemm(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW,
                int64_t lddw, const int32_t* rows, const int32_t* nrows) {
    Gemm g;   // dW[N,K] += sum_m dY[m,n] X[m,k]: both operands stored [inner][out]
    g.pass = GemmPass::WGRAD;
    g.rows = rows; g.nrows = nrows;
    g.M = N; g.N = K; g.K = M; g.A = dY; g.lda = lddy; g.B = X; g.ldb = ldx;
    g.C = dW; g.ldc = lddw; g.accumulate = 2;
    return g;
}

int linear_dx(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* W, int64_t ldw,
              float* dX, int64_t lddx, cudaStream_t s, int accumulate, const float* mask, int64_t ldmask,
              const int32_t* rows, const int32_t* nrows) {
    Gemm g = dgrad_gemm(M, N, K, dY, lddy, W, ldw, dX, lddx, rows, nrows);
    g.accumulate = accumulate; g.mask = mask; g.ldmask = ldmask;
    return gemm(g, s);
}

int linear_dw(int64_t M, int64_t N, int64_t K, const float* dY, int64_t lddy, const float* X, int64_t ldx,
              float* dW, int64_t lddw, float* db, cudaStream_t s, bool relu_x, const int32_t* rows, const int32_t* nrows) {
    if (dW) {
        Gemm g = wgrad_gemm(M, N, K, dY, lddy, X, ldx, dW, lddw, rows, nrows);
        g.relu_b = relu_x;
        INTEL_TRY(gemm(g, s));
    }
    if (db) INTEL_TRY(colsum(M, N, dY, lddy, db, s));
    return INTEL_OK;
}

// ---- column sums (bias gradients): out[n] += sum_m X[m, n] ----
__global__ void __launch_bounds__(256) colsum_kernel(int64_t M, int64_t N, const float* X, int64_t ld, float* out,
                                                     int64_t rows_per_block) {
    __shared__ float red[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t n = (int64_t)blockIdx.x * 32 + tx;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
    const int64_t r1 = (r0 + rows_per_block < M) ? r0 + rows_per_block : M;
    float acc = 0.f;
    if (n < N)
        for (int64_t r = r0 + ty; r < r1; r += 8) acc += X[r * ld + n];
    red[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i][tx];
        atomicAdd(out + n, t);
    }
}

int colsum(int64_t M, int64_t N, const float* X, int64_t ld, float* out, cudaStream_t s) {
    if (M <= 0 || N <= 0) return INTEL_OK;
    int64_t col_blocks = ceil_div(N, 32);
    int64_t want_rows = ceil_div(4 * kNumSMs, col_blocks);
    int64_t row_blocks = ceil_div(M, 64);
    if (row_blocks > want_rows) row_blocks = want_rows;
    if (row_blocks < 1) row_blocks = 1;
    int64_t rpb = ceil_div(M, row_blocks);
    row_blocks = ceil_div(M, rpb);
    dim3 grid((unsigned)col_blocks, (unsigned)row_blocks);
    LAUNCH(colsum_kernel, grid, dim3(256), 0, s, M, N, X, ld, out, rpb);
    return check_launch("colsum", 4.0 * M * N, (double)M * N);
}

}  // namespace intel
