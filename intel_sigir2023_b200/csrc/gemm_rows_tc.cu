// Persistent, warp-specialised tcgen05 GEMM for the tall products whose weight operand fits in shared memory:
//   C[M, N] = A[M, K] W^T (+ bias)   with M in the tens of thousands and N * K <= 24576 (the GRU input projections
//   [B*H, 48..64] x [384, 48..64]^T of GeneralSeq.py:64-70 and their input gradients [B*H, 384] x [384, 48..64]).
// These products are HBM streams (one pass over A and C); the generic kernel (gemm_umma.cuh) re-splits the weights in every
// CTA and runs load -> convert -> MMA -> epilogue back to back per tile.  Here
//   * the weights are split into TF32 hi / lo K-major planes ONCE per CTA and stay resident (<= 192 KB);
//   * a CTA loops over 128-row tiles with three roles that only meet at mbarriers:
//       warps 0-3  producers : thread t loads row t of the tile, splits it and stores hi / lo straight into tensor memory
//                              (the A operand is read from TMEM: no shared-memory staging of A at all), 2 buffers;
//       warp  8    issuer    : one elected lane issues the 3xTF32 tcgen05.mma chains, tcgen05.commit frees the A buffer /
//                              publishes the accumulator (2 accumulator buffers of 128 columns);
//       warps 4-7  epilogue  : tcgen05.ld -> + bias -> per-warp 4 KB transposing stage -> 128-byte coalesced row segments.
//     so the epilogue of one 128 x 128 block overlaps the MMAs of the next and the loads of the tile after.
// Two shapes of loop: several N-blocks per tile from one A buffer (forward: K <= 64), or several K-chunks accumulating into
// one block (input gradient: N <= 128).
#include "kernels.h"
#include "mma.cuh"
#ifndef INTEL_EMU
#include "tc05.cuh"

namespace intel {

namespace {
constexpr int RT_KC = 64;                 // columns of A per tensor-memory buffer (hi 64 | lo 64)
constexpr int RT_NB = 128;                // accumulator block
constexpr int RT_THREADS = 288;
constexpr int RT_GK = 2;                  // K chunks accumulated in tensor memory before the block is folded into registers

struct RowsArgs {
    int64_t M;
    int N, K;                             // K: inner dimension
    const float* A; int64_t lda;
    const float* W; int64_t ldw; int w_t;  // w_t = 0: W stored [N][K]; 1: stored [K][N]
    const float* bias;
    float* C; int64_t ldc;
    int nkc, nnc;                         // K chunks of RT_KC, N blocks of RT_NB (one of them is 1)
    const int32_t* rows;                  // optional: the rows of A / C to process (Gemm::rows), *nrows of them
    const int32_t* nrows;
};
}  // namespace

__global__ void __launch_bounds__(RT_THREADS, 1) gemm_rows_tc_kernel(RowsArgs a) {
    extern __shared__ __align__(1024) uint8_t rsm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Kp = a.nkc * RT_KC;                                   // padded inner dimension of the planes
    const int Np = (a.N + 15) / 16 * 16;
    const int plane = Np * Kp * 4;                                   // bytes of one plane [Kp / 4][Np][4]
    uint8_t* w_hi = rsm;
    uint8_t* w_lo = rsm + plane;
    float* stage = reinterpret_cast<float*>(rsm + 2 * plane);        // 4 warps x [32][32] floats
    float* bias_s = stage + 4 * 1024;                                // [Np]
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + ((Np + 31) / 32) * 32);      // a_full[2] a_empty[2] d_full[2] d_empty[2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
    // ---- weights -> resident hi / lo planes (zero padded), bias ----
    // one 16-byte plane unit (row n, 4 consecutive k) per iteration: a float4 of a [N][K] weight row, or four coalesced scalars
    // of a [K][N] one; consecutive threads take consecutive n so the shared-memory stores of a warp are contiguous
    {
        const int units = Np * (Kp / 4);
#pragma unroll 4
        for (int e = tid; e < units; e += RT_THREADS) {
            const int kq = e / Np, n = e - kq * Np, k = 4 * kq;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < a.N && k < a.K) {
                if (!a.w_t && (a.ldw % 4 == 0) && ((uintptr_t)a.W % 16 == 0)) v = *reinterpret_cast<const float4*>(a.W + (int64_t)n * a.ldw + k);
                else if (!a.w_t) v = make_float4(a.W[(int64_t)n * a.ldw + k], a.W[(int64_t)n * a.ldw + k + 1], a.W[(int64_t)n * a.ldw + k + 2],
                                                 a.W[(int64_t)n * a.ldw + k + 3]);
                else v = make_float4(a.W[(int64_t)k * a.ldw + n], a.W[(int64_t)(k + 1) * a.ldw + n], a.W[(int64_t)(k + 2) * a.ldw + n],
                                     a.W[(int64_t)(k + 3) * a.ldw + n]);
            }
            uint4 h, l;
            split_tf32(v.x, h.x, l.x);
            split_tf32(v.y, h.y, l.y);
            split_tf32(v.z, h.z, l.z);
            split_tf32(v.w, h.w, l.w);
            *reinterpret_cast<uint4*>(w_hi + (size_t)e * 16) = h;
            *reinterpret_cast<uint4*>(w_lo + (size_t)e * 16) = l;
        }
    }
    for (int n = tid; n < Np; n += RT_THREADS) bias_s[n] = (a.bias && n < a.N) ? a.bias[n] : 0.f;
    if (tid == 0) {
        tc05::mbar_init(&bars[0], 128); tc05::mbar_init(&bars[1], 128);      // a_full: the 128 producer threads
        tc05::mbar_init(&bars[2], 1); tc05::mbar_init(&bars[3], 1);          // a_empty: tcgen05.commit
        tc05::mbar_init(&bars[4], 1); tc05::mbar_init(&bars[5], 1);          // d_full: tcgen05.commit
        tc05::mbar_init(&bars[6], 128); tc05::mbar_init(&bars[7], 128);      // d_empty: the 128 epilogue threads
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) tc05::tmem_alloc(tmem_slot, 512);
    tc05::fence_smem_to_mma();
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    const uint32_t tm = *tmem_slot;
    // with a row list the tile loop runs over the listed rows only (tile i = entries [128 i, 128 i + 128) of the list)
    int64_t Mrows = a.M;
    if (a.rows) {
        const int64_t n = *a.nrows;
        Mrows = n < 0 ? 0 : (n > a.M ? a.M : n);
    }
    const int64_t tiles = (Mrows + 127) / 128;
    uint64_t *a_full = bars, *a_empty = bars + 2, *d_full = bars + 4, *d_empty = bars + 6;
    const uint32_t cA = 0, cD = 256;                                 // A buffers: 2 x (64 hi | 64 lo); accumulators: 2 x 128

    if (warp < 4) {
        // ================= producers =================
        const uint32_t tl = tm + ((uint32_t)(warp * 32) << 16);
        // the loads of chunk i + 1 (next K chunk or next tile) are issued before chunk i is split and stored, so the HBM
        // latency overlaps one chunk of work
        const int64_t my_tiles = blockIdx.x < tiles ? (tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
        const int64_t nch = my_tiles * a.nkc;
        float4 v[RT_KC / 4], nx[RT_KC / 4];
        auto load_chunk = [&](int64_t i, float4 (&x)[RT_KC / 4]) {
            const int64_t tile = blockIdx.x + (i / a.nkc) * gridDim.x;
            const int kc = (int)(i % a.nkc);
            const int64_t idx = tile * 128 + tid;
            const bool on = idx < Mrows;
            const int64_t row = (on && a.rows) ? (int64_t)a.rows[idx] : idx;
            const float* src = a.A + row * a.lda;
#pragma unroll
            for (int j = 0; j < RT_KC / 4; ++j) {
                const int k = kc * RT_KC + 4 * j;
                x[j] = (on && k < a.K) ? *reinterpret_cast<const float4*>(src + k) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        if (nch > 0) load_chunk(0, v);
        for (int64_t i = 0; i < nch; ++i) {
            const uint32_t ia = (uint32_t)i, buf = ia & 1u;
            if (i + 1 < nch) load_chunk(i + 1, nx);
            if (ia >= 2) tc05::mbar_wait(&a_empty[buf], ((ia >> 1) - 1) & 1u);
            tc05::fence_after();
#pragma unroll
            for (int q = 0; q < RT_KC / 32; ++q) {
                uint32_t h[32], lo[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    split_tf32(v[8 * q + j].x, h[4 * j], lo[4 * j]);
                    split_tf32(v[8 * q + j].y, h[4 * j + 1], lo[4 * j + 1]);
                    split_tf32(v[8 * q + j].z, h[4 * j + 2], lo[4 * j + 2]);
                    split_tf32(v[8 * q + j].w, h[4 * j + 3], lo[4 * j + 3]);
                }
                tc05::st32(tl + cA + buf * 128 + 32 * q, h);
                tc05::st32(tl + cA + buf * 128 + 64 + 32 * q, lo);
            }
            tc05::wait_st();
            tc05::fence_before();
            tc05::mbar_arrive(&a_full[buf]);
#pragma unroll
            for (int j = 0; j < RT_KC / 4; ++j) v[j] = nx[j];
        }
    } else if (warp == 8) {
        // ================= MMA issuer =================
        if (tc05::elect_one()) {
            const uint32_t lbo = (uint32_t)Np * 16;
            const uint64_t d_hi = tc05::make_desc(tc05::smem_u32(w_hi), lbo, 128), d_lo = tc05::make_desc(tc05::smem_u32(w_lo), lbo, 128);
            uint32_t ia = 0, id = 0;
            for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                if (a.nkc == 1) {                                    // forward shape: every N block from the same A buffer
                    const uint32_t ba = ia & 1u;
                    tc05::mbar_wait(&a_full[ba], (ia >> 1) & 1u);
                    for (int nc = 0; nc < a.nnc; ++nc, ++id) {
                        const uint32_t bd = id & 1u;
                        if (id >= 2) tc05::mbar_wait(&d_empty[bd], ((id >> 1) - 1) & 1u);
                        tc05::fence_after();
                        const int ncols = (Np - nc * RT_NB) < RT_NB ? (Np - nc * RT_NB) : RT_NB;
                        const uint32_t idesc = tc05::make_idesc(128, ncols);
                        const uint32_t roff = (uint32_t)(nc * RT_NB * 16);
#pragma unroll 2
                        for (int ks = 0; ks < RT_KC / 8; ++ks) {
                            const uint64_t bh = d_hi + (uint64_t)((roff + ks * 2 * lbo) >> 4), bl = d_lo + (uint64_t)((roff + ks * 2 * lbo) >> 4);
                            const uint32_t ah = tm + cA + ba * 128 + 8 * ks, al = ah + 64;
                            tc05::mma_ts(tm + cD + bd * 128, al, bh, idesc, ks ? 1u : 0u);
                            tc05::mma_ts(tm + cD + bd * 128, ah, bl, idesc, 1u);
                            tc05::mma_ts(tm + cD + bd * 128, ah, bh, idesc, 1u);
                        }
                        tc05::commit(&d_full[bd]);
                    }
                    tc05::commit(&a_empty[ba]);
                    ++ia;
                } else {                                             // input-gradient shape: K chunks accumulate into one block;
                    // the tensor core adds into the accumulator with truncation, so a block is closed after RT_GK chunks
                    // (128 inner columns) and the epilogue sums the partial blocks in fp32 registers with rounded adds
                    const uint32_t idesc = tc05::make_idesc(128, Np);
                    for (int kc = 0; kc < a.nkc; ++kc, ++ia) {
                        const uint32_t bd = id & 1u;
                        if (kc % RT_GK == 0 && id >= 2) tc05::mbar_wait(&d_empty[bd], ((id >> 1) - 1) & 1u);
                        const uint32_t ba = ia & 1u;
                        tc05::mbar_wait(&a_full[ba], (ia >> 1) & 1u);
                        tc05::fence_after();
#pragma unroll 2
                        for (int ks = 0; ks < RT_KC / 8; ++ks) {
                            const uint32_t koff = (uint32_t)((kc * (RT_KC / 4) + 2 * ks) * lbo);
                            const uint64_t bh = d_hi + (uint64_t)(koff >> 4), bl = d_lo + (uint64_t)(koff >> 4);
                            const uint32_t ah = tm + cA + ba * 128 + 8 * ks, al = ah + 64;
                            tc05::mma_ts(tm + cD + bd * 128, al, bh, idesc, ((kc % RT_GK) | ks) ? 1u : 0u);
                            tc05::mma_ts(tm + cD + bd * 128, ah, bl, idesc, 1u);
                            tc05::mma_ts(tm + cD + bd * 128, ah, bh, idesc, 1u);
                        }
                        tc05::commit(&a_empty[ba]);
                        if (kc % RT_GK == RT_GK - 1 || kc == a.nkc - 1) {
                            tc05::commit(&d_full[bd]);
                            ++id;
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else {
        // ================= epilogue =================
        const int ew = warp - 4;
        const uint32_t tl = tm + ((uint32_t)(ew * 32) << 16);
        float* st = stage + ew * 1024;
        uint32_t id = 0;
        const int groups = a.nkc > 1 ? (a.nkc + RT_GK - 1) / RT_GK : 1;
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int64_t m0 = tile * 128 + ew * 32;
            // destination row of this lane's tile row (-1: none); the store loops fetch the row of tile row r from lane r
            int64_t myrow = -1;
            if (m0 + lane < Mrows) myrow = a.rows ? (int64_t)a.rows[m0 + lane] : m0 + lane;
            if (a.nkc > 1) {
                // ---- partial blocks of one 128 x Np (<= 64) output block: summed in registers, stored once ----
                float acc[64];
#pragma unroll
                for (int j = 0; j < 64; ++j) acc[j] = 0.f;
                for (int grp = 0; grp < groups; ++grp, ++id) {
                    const uint32_t bd = id & 1u;
                    tc05::mbar_wait(&d_full[bd], (id >> 1) & 1u);
                    tc05::fence_after();
                    uint32_t u[32], v[32];
                    tc05::ld32(tl + cD + bd * 128, u);
                    if (Np > 32) tc05::ld32(tl + cD + bd * 128 + 32, v);
                    tc05::wait_ld();
                    tc05::fence_before();
                    tc05::mbar_arrive(&d_empty[bd]);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        acc[j] += __uint_as_float(u[j]);
                        if (Np > 32) acc[32 + j] += __uint_as_float(v[j]);
                    }
                }
                for (int g = 0; g < Np; g += 32) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float4 v4;
                        if (g == 0) v4 = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
                        else v4 = make_float4(acc[32 + 4 * j], acc[32 + 4 * j + 1], acc[32 + 4 * j + 2], acc[32 + 4 * j + 3]);
                        *reinterpret_cast<float4*>(st + lane * 32 + ((j + lane) & 7) * 4) = v4;
                    }
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int r = 4 * i + (lane >> 3), ch = lane & 7;
                        const float4 v4 = *reinterpret_cast<const float4*>(st + r * 32 + ((ch + r) & 7) * 4);
                        const int64_t row = __shfl_sync(0xffffffffu, myrow, r);
                        const int col = g + 4 * ch;
                        if (row >= 0 && col < a.N) *reinterpret_cast<float4*>(a.C + row * a.ldc + col) = v4;
                    }
                    __syncwarp();
                }
                continue;
            }
            for (int nc = 0; nc < a.nnc; ++nc, ++id) {
                const uint32_t bd = id & 1u;
                tc05::mbar_wait(&d_full[bd], (id >> 1) & 1u);
                tc05::fence_after();
                const int ncols = (Np - nc * RT_NB) < RT_NB ? (Np - nc * RT_NB) : RT_NB;
                for (int g = 0; g < ncols; g += 32) {
                    uint32_t u[32];
                    if (ncols - g >= 32) tc05::ld32(tl + cD + bd * 128 + g, u);
                    else {
                        uint32_t u16[16];
                        tc05::ld16(tl + cD + bd * 128 + g, u16);
#pragma unroll
                        for (int j = 0; j < 16; ++j) { u[j] = u16[j]; u[16 + j] = 0u; }
                    }
                    tc05::wait_ld();
                    const int n0 = nc * RT_NB + g;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {                     // own row -> stage, 16-byte chunks rotated by the row
                        float4 v;
                        v.x = __uint_as_float(u[4 * j]) + bias_s[n0 + 4 * j];
                        v.y = __uint_as_float(u[4 * j + 1]) + bias_s[n0 + 4 * j + 1];
                        v.z = __uint_as_float(u[4 * j + 2]) + bias_s[n0 + 4 * j + 2];
                        v.w = __uint_as_float(u[4 * j + 3]) + bias_s[n0 + 4 * j + 3];
                        *reinterpret_cast<float4*>(st + lane * 32 + ((j + lane) & 7) * 4) = v;
                    }
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {                     // 4 rows x 128 contiguous bytes per instruction
                        const int r = 4 * i + (lane >> 3), ch = lane & 7;
                        const float4 v = *reinterpret_cast<const float4*>(st + r * 32 + ((ch + r) & 7) * 4);
                        const int64_t row = __shfl_sync(0xffffffffu, myrow, r);
                        const int col = n0 + 4 * ch;
                        if (row >= 0 && col < a.N) *reinterpret_cast<float4*>(a.C + row * a.ldc + col) = v;
                    }
                    __syncwarp();
                }
                tc05::fence_before();
                tc05::mbar_arrive(&d_empty[bd]);
            }
        }
    }
    tc05::fence_before();
    __syncthreads();
    if (warp == 8) tc05::tmem_free(tm, 512);
}

// returns true when the product was taken (status = launch status)
bool gemm_rows_tc_try(const Gemm& g, cudaStream_t s, int* status) {
    if (g.pass == GemmPass::WGRAD || g.relu_a || g.relu_b || g.relu_out || g.add || g.mask || g.accumulate != 0) return false;
    if (g.M < 16384 || g.N < 16 || g.N % 4 || g.K % 4 || g.lda % 4 || g.ldc % 4) return false;
    if ((((uintptr_t)g.A) | ((uintptr_t)g.C)) % 16) return false;
    if (g.pass == GemmPass::DGRAD && g.bias) return false;
    const int Np = (int)((g.N + 15) / 16 * 16);
    const int nkc = (int)((g.K + RT_KC - 1) / RT_KC), nnc = (Np + RT_NB - 1) / RT_NB;
    if (nkc > 1 && (nnc > 1 || Np > 64)) return false;
    const size_t plane = (size_t)Np * nkc * RT_KC * 4;
    const size_t smem = 2 * plane + 4 * 4096 + (size_t)((Np + 31) / 32 * 32) * 4 + 128;
    if (smem > 225 * 1024) return false;
    if (!status) return true;
    RowsArgs a;
    a.M = g.M; a.N = (int)g.N; a.K = (int)g.K; a.A = g.A; a.lda = g.lda; a.W = g.B; a.ldw = g.ldb; a.w_t = g.pass == GemmPass::DGRAD;
    a.bias = g.bias; a.C = g.C; a.ldc = g.ldc; a.nkc = nkc; a.nnc = nnc;
    a.rows = (g.rows && g.nrows) ? g.rows : nullptr; a.nrows = g.nrows;
    ensure_smem(gemm_rows_tc_kernel, smem);
    const unsigned grid = stream_grid((g.M + 127) / 128, 1);
    LAUNCH(gemm_rows_tc_kernel, dim3(grid), dim3(RT_THREADS), smem, s, a);
    *status = gemm_check_launch(g, "rows_tc");
    return true;
}

}  // namespace intel
#endif
