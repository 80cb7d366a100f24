// GRU recurrence of GRU4RecEncoder (GeneralSeq.py:58-78, nn.GRU(hidden 128)) on the 5th-generation tensor cores.
//
// One thread-block CLUSTER of four CTAs owns a tile of 128 sessions for all T steps.  CTA c of the cluster owns the hidden
// units [32 c, 32 c + 32): its 96 rows of W_hh (r | z | n gates of those units) stay resident in shared memory as pre-split
// TF32 hi / lo planes (96 KB) - the UMMA B operand of every step - and its 128 threads each own one session row (= one TMEM
// lane).  Per step:
//   h_{t-1} (all 128 units of the row, fp32, from the cluster-shared staging tile) -> hi / lo planes in tensor memory
//   gh = h_{t-1} W_hh[own rows]^T : 16 k-slices x 3 tcgen05.mma (3xTF32), M = 128 sessions, N = 96, accumulator in TMEM
//   gates of the 32 own units on the row (tcgen05.ld), h_t slice -> h_all / gates in HBM, and into the staging tile of all
//   four CTAs through distributed shared memory (st.shared::cluster), two cluster barriers per step.
// The mma.sync kernel (gru.cu) re-splits W_hh from fp32 shared memory in every step and runs 32 sessions per CTA; here the
// split happens once per launch and a step is 48 MMAs + ~100 thread-local instructions per unit.
#include "kernels.h"
#include "mma.cuh"
#ifndef INTEL_EMU
#include "tc05.cuh"

namespace intel {

namespace {
constexpr int GT_H = 128, GT_U = 32, GT_N = 96;                  // hidden, units per CTA, gate rows per CTA
constexpr int GT_W_LBO = GT_N * 16;                              // W planes [k-chunk (32)][96 rows][4]
constexpr int GT_W_HI = 0, GT_W_LO = 49152, GT_STAGE = 98304;    // staging tile [128 rows][32 chunks of 16 B], chunk index rotated by row
constexpr int GT_BIAS = GT_STAGE + 65536, GT_BAR = GT_BIAS + 512, GT_TMEM = GT_BAR + 16, GT_BYTES = GT_BAR + 64;

__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
// arrival without the release fence (which would wait for every global store still in flight): used where the arrival only
// says "my reads of the shared tile are done"
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, float a, float b, float c, float d) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float ex2a(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcpa(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sigmoid / tanh from MUFU.EX2 + MUFU.RCP (relative error ~2^-21 of the exponential; the results feed fp32 sums whose
// parity budget is 1e-5 of the tensor's largest entry)
__device__ __forceinline__ float sigmoid_fast(float x) { return rcpa(1.0f + ex2a(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return 1.0f - 2.0f * rcpa(1.0f + ex2a(2.885390081777927f * x)); }
}  // namespace

// Up to two encoders (the session-history and the item-history GRU of IntEL.predict_intent) share one launch: cluster q
// serves encoder q % nenc, tile q / nenc.  With the length-sorted session order of each encoder (longest first) the hardware
// hands out the clusters in blockIdx order = by decreasing length of both encoders interleaved, a cluster stops at the last
// live step of its tile, and the SMs it frees take the next cluster: the two recurrences, each a chain of T dependent steps,
// overlap instead of running back to back.
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(128, 1) gru_tc_fwd_kernel(GruTcPair args) {
    extern __shared__ __align__(1024) uint8_t gsm[];
    const int t = threadIdx.x, warp = t >> 5;
    const uint32_t c = cluster_rank();                              // hidden-unit slice of this CTA
    const int cq = (int)(blockIdx.x >> 2);
    const GruTcOne& E = args.e[cq % args.n];
    const int64_t tile = cq / args.n;
    const int64_t B = E.B, T = E.T;
    if (tile * 128 >= B) return;                                     // the whole cluster leaves (no barrier was touched)
    const int64_t* __restrict__ lens = E.lens;
    const float* __restrict__ gi = E.gi;
    const float* __restrict__ w_hh = E.w_hh;
    const float* __restrict__ b_hh = E.b_hh;
    float* __restrict__ h_all = E.h_all;
    float* __restrict__ gates = E.gates;
    const int save_gates = args.save_gates;
    const int64_t slot = tile * 128 + t;
    const int64_t b = slot < B ? (E.order ? (int64_t)E.order[slot] : slot) : B;      // this thread's session (B: none)
    // the tile's loop bound: the longest session comes first in the sorted order (same value in all four CTAs)
    int64_t tmax = T;
    if (E.order) {
        const int64_t l0 = lens[E.order[tile * 128]];
        tmax = l0 < 0 ? 0 : (l0 > T ? T : l0);
    }
    uint64_t* bar = reinterpret_cast<uint64_t*>(gsm + GT_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gsm + GT_TMEM);
    float* bias = reinterpret_cast<float*>(gsm + GT_BIAS);           // [3][32] of the own units
    // ---- W_hh rows of the own units -> hi / lo planes (plane row = gate * 32 + unit) ----
    // one 16-byte plane unit (row n, 4 consecutive k) per iteration = one float4 of a W_hh row
#pragma unroll 4
    for (int e = t; e < GT_N * (GT_H / 4); e += 128) {
        const int kq = e / GT_N, n = e - kq * GT_N;
        const int grow = (n >> 5) * GT_H + (int)c * GT_U + (n & 31);
        const float4 v = *reinterpret_cast<const float4*>(w_hh + grow * GT_H + 4 * kq);
        uint4 h, l;
        split_tf32(v.x, h.x, l.x);
        split_tf32(v.y, h.y, l.y);
        split_tf32(v.z, h.z, l.z);
        split_tf32(v.w, h.w, l.w);
        *reinterpret_cast<uint4*>(gsm + GT_W_HI + (size_t)e * 16) = h;
        *reinterpret_cast<uint4*>(gsm + GT_W_LO + (size_t)e * 16) = l;
    }
    if (t < GT_N) bias[t] = b_hh[(t >> 5) * GT_H + (int)c * GT_U + (t & 31)];
    for (int e = t; e < 128 * 32; e += 128) reinterpret_cast<uint4*>(gsm + GT_STAGE)[e] = make_uint4(0u, 0u, 0u, 0u);      // h_0 = 0
    if (t == 0) {
        tc05::mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (t < 32) tc05::tmem_alloc(tmem_slot, 512);
    tc05::fence_smem_to_mma();
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    const uint32_t tm = *tmem_slot;
    const uint32_t tl = tm + ((uint32_t)(warp * 32) << 16);
    const uint32_t cHi = 0, cLo = 128, cD = 256;
    const uint64_t d_hi = tc05::make_desc(tc05::smem_u32(gsm + GT_W_HI), GT_W_LBO, 128);
    const uint64_t d_lo = tc05::make_desc(tc05::smem_u32(gsm + GT_W_LO), GT_W_LBO, 128);
    const uint32_t idesc = tc05::make_idesc(128, GT_N);
    const uint32_t stage_local = tc05::smem_u32(gsm + GT_STAGE);
    uint32_t stage_remote[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) stage_remote[q] = map_to_cta(stage_local, (uint32_t)q);
    const int64_t len = b < B ? lens[b] : 0;
    float hp[GT_U];                                                  // own units of h_{t-1}
#pragma unroll
    for (int u = 0; u < GT_U; ++u) hp[u] = 0.f;
    uint32_t phase = 0;
    cluster_arrive();                                                // every CTA of the cluster has zeroed its staging tile
    cluster_wait();

    for (int64_t ts = 0; ts < tmax; ++ts) {
        const bool live = ts < len;
        const float* gin = gi + (b * T + ts) * 3 * GT_H + (int)c * GT_U;
        // ---- h_{t-1} of the row: staging tile -> hi / lo planes in tensor memory ----
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t h[32], lo[32];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 v = *reinterpret_cast<const float4*>(gsm + GT_STAGE + t * 512 + ((8 * q + j + t) & 31) * 16);
                split_tf32(v.x, h[4 * j], lo[4 * j]);
                split_tf32(v.y, h[4 * j + 1], lo[4 * j + 1]);
                split_tf32(v.z, h[4 * j + 2], lo[4 * j + 2]);
                split_tf32(v.w, h[4 * j + 3], lo[4 * j + 3]);
            }
            tc05::st32(tl + cHi + 32 * q, h);
            tc05::st32(tl + cLo + 32 * q, lo);
        }
        cluster_arrive_relaxed();                                    // (A) this CTA is done reading its staging tile
        tc05::wait_st();
        tc05::fence_before();
        __syncthreads();
        if (warp == 0) {
            tc05::fence_after();
            if (tc05::elect_one()) {
#pragma unroll 4
                for (int ks = 0; ks < GT_H / 8; ++ks) {
                    const uint64_t bh = d_hi + (uint64_t)((ks * 2 * GT_W_LBO) >> 4), bl = d_lo + (uint64_t)((ks * 2 * GT_W_LBO) >> 4);
                    tc05::mma_ts(tm + cD, tm + cLo + 8 * ks, bh, idesc, ks ? 1u : 0u);
                    tc05::mma_ts(tm + cD, tm + cHi + 8 * ks, bl, idesc, 1u);
                    tc05::mma_ts(tm + cD, tm + cHi + 8 * ks, bh, idesc, 1u);
                }
                tc05::commit(bar);
            }
            __syncwarp();
        }
        // this step's input pre-activations travel while the product runs
        float4 gv[3][8];
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int j = 0; j < 8; ++j) gv[g][j] = live ? *reinterpret_cast<const float4*>(gin + g * GT_H + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        tc05::mbar_wait(bar, phase);
        phase ^= 1u;
        tc05::fence_after();
        // ---- gates of the own units ----
        float rr[GT_U], zz[GT_U], nn[GT_U], gg[GT_U];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            uint32_t dr[16], dz[16], dn[16];
            tc05::ld16(tl + cD + 16 * half, dr);
            tc05::ld16(tl + cD + 32 + 16 * half, dz);
            tc05::ld16(tl + cD + 64 + 16 * half, dn);
            tc05::wait_ld();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int u = 16 * half + j;
                const float4 a4 = gv[0][u >> 2], b4 = gv[1][u >> 2], c4 = gv[2][u >> 2];
                const float ir = (u & 3) == 0 ? a4.x : ((u & 3) == 1 ? a4.y : ((u & 3) == 2 ? a4.z : a4.w));
                const float iz = (u & 3) == 0 ? b4.x : ((u & 3) == 1 ? b4.y : ((u & 3) == 2 ? b4.z : b4.w));
                const float in = (u & 3) == 0 ? c4.x : ((u & 3) == 1 ? c4.y : ((u & 3) == 2 ? c4.z : c4.w));
                rr[u] = sigmoid_fast(ir + __uint_as_float(dr[j]) + bias[u]);
                zz[u] = sigmoid_fast(iz + __uint_as_float(dz[j]) + bias[32 + u]);
                gg[u] = __uint_as_float(dn[j]) + bias[64 + u];
                nn[u] = tanh_fast(in + rr[u] * gg[u]);
                if (live) hp[u] = (1.f - zz[u]) * nn[u] + zz[u] * hp[u];
            }
        }
        cluster_wait();                                              // (A) every CTA has read h_{t-1}: the tiles may be overwritten
        // ---- h_t slice into every CTA's staging tile first: the release fence of the arrival then only has these
        //      shared-memory stores to wait for; the HBM stores follow and overlap the barrier ----
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t off = (uint32_t)(t * 512 + ((8 * (int)c + j + t) & 31) * 16);
#pragma unroll
            for (int q = 0; q < 4; ++q) st_cluster_v4(stage_remote[q] + off, hp[4 * j], hp[4 * j + 1], hp[4 * j + 2], hp[4 * j + 3]);
        }
        cluster_arrive();                                            // (B) h_t is in every staging tile
        if (b < B) {
            float* ho = h_all + (b * (T + 1) + ts + 1) * GT_H + (int)c * GT_U;
#pragma unroll
            for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(ho + 4 * j) = make_float4(hp[4 * j], hp[4 * j + 1], hp[4 * j + 2], hp[4 * j + 3]);
        }
        if (live && save_gates) {
            float* gt = gates + (b * T + ts) * 4 * GT_H + (int)c * GT_U;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                *reinterpret_cast<float4*>(gt + 4 * j) = make_float4(rr[4 * j], rr[4 * j + 1], rr[4 * j + 2], rr[4 * j + 3]);
                *reinterpret_cast<float4*>(gt + GT_H + 4 * j) = make_float4(zz[4 * j], zz[4 * j + 1], zz[4 * j + 2], zz[4 * j + 3]);
                *reinterpret_cast<float4*>(gt + 2 * GT_H + 4 * j) = make_float4(nn[4 * j], nn[4 * j + 1], nn[4 * j + 2], nn[4 * j + 3]);
                *reinterpret_cast<float4*>(gt + 3 * GT_H + 4 * j) = make_float4(gg[4 * j], gg[4 * j + 1], gg[4 * j + 2], gg[4 * j + 3]);
            }
        }
        cluster_wait();
    }
    // a tile that stopped early: the final state goes to slot T (the output projection reads it there), the slots between
    // are cleared (only weight-gradient paths that ignore the live-row list read them, against zero gradient rows)
    if (tmax < T && b < B) {
        for (int64_t ts = tmax + 1; ts <= T; ++ts) {
            float* ho = h_all + (b * (T + 1) + ts) * GT_H + (int)c * GT_U;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                *reinterpret_cast<float4*>(ho + 4 * j) = ts == T ? make_float4(hp[4 * j], hp[4 * j + 1], hp[4 * j + 2], hp[4 * j + 3])
                                                                 : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    tc05::fence_before();
    __syncthreads();
    if (t < 32) tc05::tmem_free(tm, 512);
    cluster_arrive();                                                // no CTA leaves while a peer may still write into it
    cluster_wait();
}

static int g_use_gru_tc = 1;
void gru_debug_use_tcgen05(int on) { g_use_gru_tc = on ? 1 : 0; }
bool gru_tc_supported() { return g_use_gru_tc; }

int gru_tc_fwd_pair(const GruTcPair& p, cudaStream_t s) {
    int64_t tiles = 0;
    double bytes = 0.0, flops = 0.0;
    for (int i = 0; i < p.n; ++i) {
        const GruTcOne& o = p.e[i];
        const int64_t ti = ceil_div(o.B, 128);
        tiles = ti > tiles ? ti : tiles;
        bytes += (double)o.B * o.T * (3 + (p.save_gates ? 4 : 0) + 1) * GT_H * 4.0;
        flops += 2.0 * o.B * o.T * 3 * GT_H * GT_H;
    }
    if (tiles <= 0) return INTEL_OK;
    const unsigned grid = (unsigned)(4 * tiles * p.n);
    ensure_smem(gru_tc_fwd_kernel, (size_t)GT_BYTES);
    LAUNCH(gru_tc_fwd_kernel, dim3(grid), dim3(128), (size_t)GT_BYTES, s, p);
    return check_launch("gru_seq_fwd", bytes, flops);
}

}  // namespace intel
#else
namespace intel {
void gru_debug_use_tcgen05(int) {}
bool gru_tc_supported() { return false; }
int gru_tc_fwd_pair(const GruTcPair&, cudaStream_t) { return INTEL_ERR_UNSUPPORTED; }
}  // namespace intel
#endif
