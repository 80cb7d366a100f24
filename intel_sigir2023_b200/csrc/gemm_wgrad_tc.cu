// Weight gradients of the tall nn.Linear passes on tcgen05:  dW[M, N] += sum_r dY[r, m] X[r, n]  with tens of thousands of
// rows r, M a multiple of 128 and N <= 128 (the GRU input / recurrent weights: [384 x 48..128] over 81 920..86 016 rows).
// The contraction runs over the ROWS of both operands, i.e. both are MN-major for the tensor core: a [32 rows][32 floats]
// natural tile whose 32-byte chunk index is XORed with (row & 3) is exactly the SWIZZLE_128B_BASE32B atom (probe 9 / 11 of
// tests/hw/umma_probe.cu), so the operands go from global memory to shared memory in their own row-major order, split into
// TF32 hi / lo on the way, with 16-byte stores that fill 512 contiguous bytes per warp instruction.
//
// A CTA owns a 128-column slice of dY, all N columns of X and a contiguous range of rows (split-K over the grid, fp32 atomics at
// the end).  8 worker warps load + split 32-row stages into a 3-deep ring; one issuer lane runs 12 tcgen05.mma per stage
// (4 k-slices of 8 rows x 3xTF32), accumulating 128 rows per tensor-memory block (the tensor core adds with truncation: longer
// chains drift), two blocks in flight; the workers fold a finished block into fp32 registers while the next one is being fed.
#include "kernels.h"
#include "mma.cuh"
#ifndef INTEL_EMU
#include "tc05.cuh"

namespace intel {

namespace {
constexpr int WG_STAGE_ROWS = 32, WG_STAGES = 3, WG_BLOCK_STAGES = 4;
constexpr int WG_SUB = 4096;                               // bytes of one [32 rows][32 floats] sub-tile
constexpr int WG_STAGE_BYTES = 16 * WG_SUB;                // A hi 4 | A lo 4 | B hi 4 | B lo 4 sub-tiles
constexpr int WG_THREADS = 288;                            // 8 worker warps + 1 issuer warp

struct WgradArgs {
    int64_t R;                             // rows (the contraction)
    int M, N;                              // dW is [M][N]; this CTA takes columns [128 blockIdx.x, +128) of dY
    const float* dY; int64_t ldy;
    const float* X; int64_t ldx;
    float* dW; int64_t ldw;
    int64_t blocks_per_cta;                // 128-row blocks per CTA along the rows
    const int32_t* rows;                   // optional: the rows to contract over (Gemm::rows), *nrows of them
    const int32_t* nrows;
};

// byte offset of 16-byte chunk `ch` (0..7) of row `r` (0..31) inside a sub-tile: 32-byte chunk index ^ (row & 3)
__device__ __forceinline__ int sub_off(int r, int ch) { return r * 128 + ((((ch >> 1) ^ (r & 3)) << 1) | (ch & 1)) * 16; }
}  // namespace

__global__ void __launch_bounds__(WG_THREADS, 1) gemm_wgrad_tc_kernel(WgradArgs a) {
    extern __shared__ __align__(1024) uint8_t wsm[];
    __shared__ __align__(8) uint64_t bars[2 * WG_STAGES + 4];            // stage_full[3] stage_empty[3] acc_full[2] acc_empty[2]
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t *stage_full = bars, *stage_empty = bars + WG_STAGES, *acc_full = bars + 2 * WG_STAGES, *acc_empty = acc_full + 2;
    const int nsub = (a.N + 31) / 32;                                     // sub-tiles of X per stage (the last one zero padded)
    const int Np = nsub * 32;
    if (tid == 0) {
        for (int i = 0; i < WG_STAGES; ++i) { tc05::mbar_init(&stage_full[i], 256); tc05::mbar_init(&stage_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { tc05::mbar_init(&acc_full[i], 1); tc05::mbar_init(&acc_empty[i], 256); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) tc05::tmem_alloc(&tmem_slot, 256);
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    const uint32_t tm = tmem_slot;
    const int m0 = blockIdx.x * 128;
    // with a row list the contraction runs over the listed rows only; the split over the grid follows their number
    int64_t R = a.R, bpc = a.blocks_per_cta;
    if (a.rows) {
        const int64_t n = *a.nrows;
        R = n < 0 ? 0 : (n > a.R ? a.R : n);
        bpc = ((R + 127) / 128 + gridDim.y - 1) / gridDim.y;
    }
    const int64_t blk0 = (int64_t)blockIdx.y * bpc;
    const int64_t total_blocks = (R + 127) / 128;
    int64_t nblk = total_blocks - blk0;
    if (nblk > bpc) nblk = bpc;
    if (nblk < 0) nblk = 0;

    if (warp < 8) {
        // ================= workers: load + split stages, fold finished blocks =================
        const int half = warp >> 2;                                       // column half of the accumulator this thread folds
        const int cols = Np / 2;                                          // 16, 32 or 64
        const uint32_t tl = tm + ((uint32_t)((warp & 3) * 32) << 16);
        float acc[64];
#pragma unroll
        for (int j = 0; j < 64; ++j) acc[j] = 0.f;
        auto fold = [&](int64_t j) {
            const uint32_t buf = (uint32_t)(j & 1);
            tc05::mbar_wait(&acc_full[buf], (uint32_t)((j >> 1) & 1));
            tc05::fence_after();
            const uint32_t c0 = buf * 128 + half * cols;
            if (cols == 64) {
                uint32_t u[32], v[32];
                tc05::ld32(tl + c0, u);
                tc05::ld32(tl + c0 + 32, v);
                tc05::wait_ld();
#pragma unroll
                for (int q = 0; q < 32; ++q) { acc[q] += __uint_as_float(u[q]); acc[32 + q] += __uint_as_float(v[q]); }
            } else if (cols == 32) {
                uint32_t u[32];
                tc05::ld32(tl + c0, u);
                tc05::wait_ld();
#pragma unroll
                for (int q = 0; q < 32; ++q) acc[q] += __uint_as_float(u[q]);
            } else {
                uint32_t u[16];
                tc05::ld16(tl + c0, u);
                tc05::wait_ld();
#pragma unroll
                for (int q = 0; q < 16; ++q) acc[q] += __uint_as_float(u[q]);
            }
            tc05::fence_before();
            tc05::mbar_arrive(&acc_empty[buf]);
        };
        // unit u of a stage = (operand, sub-tile, row quad): a warp instruction moves 4 rows x 128 bytes of one sub-tile; warp w
        // takes row quad w of every sub-tile.  The loads of stage i + 1 are issued before stage i is converted, so the HBM
        // latency is covered by one stage of work instead of being paid per stage.
        const int units_b = nsub * 8;
        const int r = 4 * warp + (lane >> 3), ch = lane & 7;
        const int64_t nst = nblk * WG_BLOCK_STAGES;
        float4 va[4], vb[4], na[4], nb[4];
        auto load_stage = [&](int64_t it, float4 (&xa)[4], float4 (&xb)[4]) {
            const int64_t idx = (blk0 * WG_BLOCK_STAGES + it) * WG_STAGE_ROWS + r;
            const bool on = idx < R;
            const int64_t row = (on && a.rows) ? (int64_t)a.rows[idx] : idx;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                xa[i] = on ? *reinterpret_cast<const float4*>(a.dY + row * a.ldy + m0 + 32 * i + 4 * ch) : make_float4(0.f, 0.f, 0.f, 0.f);
                const int col = 32 * i + 4 * ch;
                xb[i] = (i < nsub && on && col < a.N) ? *reinterpret_cast<const float4*>(a.X + row * a.ldx + col) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        if (nst > 0) load_stage(0, va, vb);
        for (int64_t it = 0; it < nst; ++it) {
            const uint32_t sc = (uint32_t)it, st = sc % WG_STAGES;
            if (it + 1 < nst) load_stage(it + 1, na, nb);
            if (sc >= WG_STAGES) tc05::mbar_wait(&stage_empty[st], ((sc / WG_STAGES) - 1) & 1u);
            uint8_t* base = wsm + st * WG_STAGE_BYTES;
            const int off0 = sub_off(r, ch);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                uint4 h, l;
                split_tf32(va[i].x, h.x, l.x); split_tf32(va[i].y, h.y, l.y); split_tf32(va[i].z, h.z, l.z); split_tf32(va[i].w, h.w, l.w);
                *reinterpret_cast<uint4*>(base + i * WG_SUB + off0) = h;
                *reinterpret_cast<uint4*>(base + (4 + i) * WG_SUB + off0) = l;
                if (i < nsub) {
                    split_tf32(vb[i].x, h.x, l.x); split_tf32(vb[i].y, h.y, l.y); split_tf32(vb[i].z, h.z, l.z); split_tf32(vb[i].w, h.w, l.w);
                    *reinterpret_cast<uint4*>(base + (8 + i) * WG_SUB + off0) = h;
                    *reinterpret_cast<uint4*>(base + (12 + i) * WG_SUB + off0) = l;
                }
            }
            tc05::fence_smem_to_mma();
            tc05::mbar_arrive(&stage_full[st]);
#pragma unroll
            for (int i = 0; i < 4; ++i) { va[i] = na[i]; vb[i] = nb[i]; }
            if ((it & 3) == 3 && it >= 7) fold((it >> 2) - 1);          // block (it / 4) is fed: fold the one before it
        }
        (void)units_b;
        if (nblk > 0) fold(nblk - 1);
        // ---- this CTA's partial sum -> dW (split-K over the grid: fp32 atomics) ----
        const int m = m0 + (warp & 3) * 32 + lane;
        if (m < a.M) {
#pragma unroll
            for (int q = 0; q < 64; ++q) {
                const int n = half * cols + q;
                if (q < cols && n < a.N) atomicAdd(a.dW + (int64_t)m * a.ldw + n, acc[q]);
            }
        }
    } else {
        // ================= MMA issuer =================
        if (tc05::elect_one()) {
            const uint32_t idesc = tc05::make_idesc(128, Np, 1, 1);
            uint32_t sc = 0;
            for (int64_t blk = 0; blk < nblk; ++blk) {
                const uint32_t buf = (uint32_t)(blk & 1);
                if (blk >= 2) tc05::mbar_wait(&acc_empty[buf], (uint32_t)(((blk >> 1) - 1) & 1));
                for (int s4 = 0; s4 < WG_BLOCK_STAGES; ++s4, ++sc) {
                    const uint32_t st = sc % WG_STAGES;
                    tc05::mbar_wait(&stage_full[st], (sc / WG_STAGES) & 1u);
                    tc05::fence_after();
                    const uint32_t base = tc05::smem_u32(wsm + st * WG_STAGE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t ah = tc05::make_desc(base + ks * 1024, WG_SUB, 512, 1), al = tc05::make_desc(base + 4 * WG_SUB + ks * 1024, WG_SUB, 512, 1);
                        const uint64_t bh = tc05::make_desc(base + 8 * WG_SUB + ks * 1024, WG_SUB, 512, 1),
                                       bl = tc05::make_desc(base + 12 * WG_SUB + ks * 1024, WG_SUB, 512, 1);
                        tc05::mma_ss(tm + buf * 128, al, bh, idesc, (s4 | ks) ? 1u : 0u);
                        tc05::mma_ss(tm + buf * 128, ah, bl, idesc, 1u);
                        tc05::mma_ss(tm + buf * 128, ah, bh, idesc, 1u);
                    }
                    tc05::commit(&stage_empty[st]);
                }
                tc05::commit(&acc_full[buf]);
            }
        }
        __syncwarp();
    }
    tc05::fence_before();
    __syncthreads();
    if (warp == 8) tc05::tmem_free(tm, 256);
}

// dW[M, N] += dY^T X (both stored [rows][cols]); false = shape not taken
bool gemm_wgrad_tc_try(const Gemm& g, cudaStream_t s, int* status) {
    if (g.pass != GemmPass::WGRAD || g.accumulate != 2 || g.relu_a || g.relu_b || g.relu_out || g.add || g.mask || g.bias) return false;
    if (g.M < 128 || g.M % 128 || g.N < 32 || g.N > 128 || g.N % 4 || g.K < 16384) return false;
    if (g.lda % 4 || g.ldb % 4 || (((uintptr_t)g.A) | ((uintptr_t)g.B)) % 16) return false;
    const int nsub = (int)((g.N + 31) / 32);
    if (nsub == 3) return false;                                          // N padded to 96: the fold assumes 32 / 64 / 128 columns
    if (!status) return true;
    WgradArgs a;
    a.R = g.K; a.M = (int)g.M; a.N = (int)g.N; a.dY = g.A; a.ldy = g.lda; a.X = g.B; a.ldx = g.ldb; a.dW = g.C; a.ldw = g.ldc;
    a.rows = (g.rows && g.nrows) ? g.rows : nullptr; a.nrows = g.nrows;
    const int mslices = (int)(g.M / 128);
    const int64_t blocks = (g.K + 127) / 128;
    int64_t splits = kNumSMs / mslices;
    if (splits < 1) splits = 1;
    if (splits > blocks) splits = blocks;
    a.blocks_per_cta = (blocks + splits - 1) / splits;
    splits = (blocks + a.blocks_per_cta - 1) / a.blocks_per_cta;
    const size_t smem = (size_t)WG_STAGES * WG_STAGE_BYTES + 1024;
    ensure_smem(gemm_wgrad_tc_kernel, smem);
    LAUNCH(gemm_wgrad_tc_kernel, dim3((unsigned)mslices, (unsigned)splits), dim3(WG_THREADS), smem, s, a);
    *status = gemm_check_launch(g, "wgrad_tc");
    return true;
}

}  // namespace intel
#endif
