// tcgen05 (5th-generation tensor core) path of the fp32-parity GEMM, included by gemm.cu.
//
// One CTA (256 threads) owns a 128 x BN output tile whose accumulator lives in tensor memory (TMEM).
//   1. cp.async streams the raw fp32 k-tiles (16 wide) of both operands into a ring of shared-memory stages,
//      NRAW - 1 tiles ahead of their use, so the HBM latency is covered by the ring and not by occupancy;
//   2. every thread converts the chunks it copied itself (no barrier needed): each value is split into its TF32
//      hi / lo parts, written as two planes per operand in the UMMA no-swizzle K-major canonical form (8 x 16-byte
//      core matrices).  An operand stored [K][rows] is transposed on the way: a thread owns a 4 x 4 block;
//   3. one elected thread issues three tcgen05.mma.kind::tf32 per 8-wide k-slice (lo*hi, hi*lo, hi*hi - the
//      3xTF32 product) that accumulate into the same TMEM tile.  MMAs run asynchronously: a tcgen05.commit on an
//      mbarrier frees the plane stage for the k-tile after next;
//   4. epilogue: tcgen05.ld, staging through shared memory, coalesced row stores with bias / residual / relu / mask.
// All three nn.Linear passes (forward, input gradient, weight gradient) run through this kernel.  (MN-major fp32
// operands would need the 128B_BASE32B swizzle; the transposing conversion is simpler.)
// The tensor core adds into the accumulator with truncation (see gemm_tc_kernel), so every UCH k-tiles the
// TMEM tile is drained into fp32 registers with a rounded add and the next MMA starts a fresh sum.
#pragma once
#ifndef INTEL_EMU
#include "tc05.cuh"

namespace intel {
namespace umma {

static const int UM = 128;           // tile rows = MMA M (cta_group::1)
static const int UBK = 16;           // k-tile per shared-memory stage (two k = 8 MMA slices)
static const int USTAGES = 2;          // plane stages (MMA of tile i overlaps the conversion of tile i + 1)
// raw fp32 stages filled by cp.async (prefetch distance NRAW - 1) are a template parameter: 4 for long inner
// dimensions, 2 for short ones (less shared memory, two CTAs per SM for the epilogue-dominated products)
static const int USBO = 144;           // stride of an 8-row core-matrix group: 128 + 16 keeps the transposing stores conflict-free
static const int UCH = 8;            // k-tiles per accumulation chunk (drained into registers with rounded adds)
static const int UTHREADS = 256;       // 8 warps: copy / convert work is spread over all of them, warps w and w + 4 share TMEM lanes

// Shared-memory plane of one operand and stage: ROWS x 16 TF32 words, K-major no-swizzle canonical layout:
// 16-byte unit (row r, k-chunk c) at c * LBO + (r / 8) * USBO + (r % 8) * 16;  LBO == 64 (mod 128) spreads the four
// k-chunks a warp writes over all banks
__host__ __device__ inline int lbo_k(int rows) { return (((rows / 8) * USBO - 64 + 127) / 128) * 128 + 64; }
__host__ __device__ inline int plane_bytes(int rows) { return (UBK / 4) * lbo_k(rows); }
__host__ __device__ inline int raw_bytes(int rows) { return rows * UBK * 4; }
__host__ __device__ inline int unit_off(int rows, int r, int c) { return c * lbo_k(rows) + (r >> 3) * USBO + (r & 7) * 16; }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int bytes) {      // bytes < 16: zero-filled tail
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src, int bytes) {        // bytes = 4 or 0 (zero fill)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void put_unit(uint8_t* hi, uint8_t* lo, int off, float a, float b, float c, float d, int relu) {
    if (relu) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); c = fmaxf(c, 0.f); d = fmaxf(d, 0.f); }
    uint4 h, l;
    split_tf32(a, h.x, l.x);
    split_tf32(b, h.y, l.y);
    split_tf32(c, h.z, l.z);
    split_tf32(d, h.w, l.w);
    *reinterpret_cast<uint4*>(hi + off) = h;
    *reinterpret_cast<uint4*>(lo + off) = l;
}

// Raw stage of an operand tile: stored [rows][K]: [rows][16] (chunk e = 4 r + c at 16 e);  stored [K][rows]:
// [16][rows].  A thread copies and later converts the same chunks: chunks e = tid + 128 i, or, transposing, the
// 4 x 4 block (rows 4 q .., k 4 c ..) with q = tid % (rows / 4), c = tid / (rows / 4).  Everything that does not
// depend on the k-tile is computed once per thread:
template <bool TR>
struct Lane {
    int n;                      // chunks this thread owns (0..4)
    int raw[4];                 // byte offset of chunk j in the raw stage
    int unit[4];                // byte offset of converted unit j in a plane
    int kof[4];                 // k offset of chunk j inside the tile
    int bytes;                  // TR: valid bytes of a chunk (row tail);  else: 16 if the row exists, 0 otherwise (per chunk below)
    int rowok[4];               // !TR: row of chunk j exists
    const float* src[4];        // global address of chunk j at k-tile 0 (k offset kof[j] included)
    int64_t step;               // elements between consecutive k-tiles
    int vec;                    // chunks are 16-byte aligned in global memory (else four 4-byte copies per chunk)

    // tr_base: first thread of the 4 x 4 transposing blocks (A uses threads 0.., B threads 128.. so that both halves work)
    __device__ __forceinline__ void init(const float* P, int64_t ld, int64_t r0, int64_t rmax, int rows, int64_t kbeg, int tid,
                                         int tr_base, int vec_) {
        vec = vec_;
        n = 0;
        bytes = 16;
        if (TR) {
            step = (int64_t)UBK * ld;
            const int bt = tid - tr_base;
            if (bt >= 0 && bt < rows) {
                const int q = bt % (rows / 4), c = bt / (rows / 4);
                const int64_t gr = r0 + 4 * q, left = rmax - gr;
                bytes = left >= 4 ? 16 : (left > 0 ? (int)left * 4 : 0);
                n = 4;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    kof[j] = 4 * c + j;
                    raw[j] = (kof[j] * rows + 4 * q) * 4;
                    unit[j] = unit_off(rows, 4 * q + j, c);
                    rowok[j] = 1;
                    src[j] = bytes ? P + (kbeg + kof[j]) * ld + gr : P;
                }
            }
        } else {
            step = UBK;
            const int units = rows * (UBK / 4);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int e = tid + j * UTHREADS;
                kof[j] = 4 * (e & 3);
                raw[j] = e * 16;
                unit[j] = unit_off(rows, e >> 2, e & 3);
                rowok[j] = 0;
                src[j] = P;
                if (e < units) {
                    n = j + 1;
                    const int64_t gr = r0 + (e >> 2);
                    rowok[j] = gr < rmax;
                    if (rowok[j]) src[j] = P + gr * ld + kbeg + kof[j];
                }
            }
        }
    }
    // cp.async of this thread's chunks of k-tile t (k0 = first k of the tile)
    __device__ __forceinline__ void issue(uint32_t rawbase, int t, int64_t k0, int64_t kend) const {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < n) {
                int b;
                if (TR) b = (k0 + kof[j] < kend) ? bytes : 0;
                else {
                    const int64_t left = kend - (k0 + kof[j]);
                    b = rowok[j] ? (left >= 4 ? 16 : (left > 0 ? (int)left * 4 : 0)) : 0;
                }
                const float* p = src[j] + (b ? (int64_t)t * step : 0);
                if (vec) cp_async16(rawbase + raw[j], p, b);
                else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) cp_async4(rawbase + raw[j] + 4 * e, 4 * e < b ? p + e : p, 4 * e < b ? 4 : 0);
                }
            }
        }
    }
    // raw chunks -> hi / lo planes
    __device__ __forceinline__ void convert(const uint8_t* rw, uint8_t* hi, uint8_t* lo, int relu) const {
        if (TR) {
            if (n) {
                float4 x[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) x[j] = *reinterpret_cast<const float4*>(rw + raw[j]);
                put_unit(hi, lo, unit[0], x[0].x, x[1].x, x[2].x, x[3].x, relu);
                put_unit(hi, lo, unit[1], x[0].y, x[1].y, x[2].y, x[3].y, relu);
                put_unit(hi, lo, unit[2], x[0].z, x[1].z, x[2].z, x[3].z, relu);
                put_unit(hi, lo, unit[3], x[0].w, x[1].w, x[2].w, x[3].w, relu);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < n) {
                    const float4 x = *reinterpret_cast<const float4*>(rw + raw[j]);
                    put_unit(hi, lo, unit[j], x.x, x.y, x.z, x.w, relu);
                }
            }
        }
    }
};

// A: M x K, ATR = stored [K][M];  B: N x K, BTR = stored [K][N];  bn = N-tile (multiple of 16, <= NACC);
// NACC = TMEM columns (32, 64 or 128); MULTI: the k range spans several accumulation chunks, which are summed in
// NACC registers per thread (single-chunk launches keep the register budget small: more CTAs per SM)
template <bool ATR, bool BTR, int NACC, bool MULTI, int NRAW>
__global__ void __launch_bounds__(UTHREADS) gemm_umma_kernel(GemmDev g, int bn, int vec_c4) {
    extern __shared__ __align__(128) uint8_t umma_smem[];
    __shared__ __align__(8) uint64_t empty_bar[USTAGES];
    __shared__ __align__(8) uint64_t chunk_bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t m0 = (int64_t)blockIdx.x * UM, n0 = (int64_t)blockIdx.y * bn;
    const int64_t kbeg = (int64_t)blockIdx.z * g.kchunk;
    const int64_t kend = (kbeg + g.kchunk < g.K) ? kbeg + g.kchunk : g.K;
    if (kbeg >= kend) return;                         // empty split (only possible with atomic accumulation)
    const int pa = plane_bytes(UM), pb = plane_bytes(bn);
    const int stage_bytes = 2 * pa + 2 * pb;
    const int ra = raw_bytes(UM), rb = raw_bytes(bn);
    uint8_t* planes = umma_smem + NRAW * (ra + rb);
    const uint32_t raw_base = tc05::smem_u32(umma_smem);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < USTAGES; ++s) tc05::mbar_init(&empty_bar[s], 1);
        tc05::mbar_init(&chunk_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tc05::tmem_alloc(&tmem_base_s, NACC);
    tc05::fence_before();
    __syncthreads();
    tc05::fence_after();
    const uint32_t tmem_d = tmem_base_s;

    const uint32_t idesc = tc05::make_idesc(UM, bn);
    const uint32_t a_lbo = lbo_k(UM), b_lbo = lbo_k(bn);

    // warps w and w + 4 read the same 32 TMEM lanes (= output rows) and take alternate 16-column chunks
    const int lanes0 = (warp & 3) * 32, chalf = warp >> 2;
    float acc[MULTI ? NACC / 2 : 1];
#pragma unroll
    for (int j = 0; j < (MULTI ? NACC / 2 : 1); ++j) acc[j] = 0.f;
    const int nk = (int)((kend - kbeg + UBK - 1) / UBK);
    uint32_t chunk_phase = 0;
    Lane<ATR> la;
    Lane<BTR> lb;
    la.init(g.A, g.lda, m0, g.M, UM, kbeg, tid, 0, g.vec_a);
    lb.init(g.B, g.ldb, n0, g.N, bn, kbeg, tid, UTHREADS / 2, g.vec_b);
    // prologue: the first NRAW - 1 k-tiles are on their way (one cp.async group per tile, empty groups keep the count uniform)
#pragma unroll
    for (int p = 0; p < NRAW - 1; ++p) {
        if (p < nk) {
            const int64_t k0 = kbeg + (int64_t)p * UBK;
            la.issue(raw_base + p * (ra + rb), p, k0, kend);
            lb.issue(raw_base + p * (ra + rb) + ra, p, k0, kend);
        }
        cp_async_commit();
    }
    for (int i = 0; i < nk; ++i) {
        const int s = i % USTAGES;
        uint8_t* st = planes + s * stage_bytes;
        cp_async_wait<NRAW - 2>();                                                        // this thread's chunks of k-tile i have landed
        if (i >= USTAGES) tc05::mbar_wait(&empty_bar[s], (uint32_t)((i / USTAGES) - 1) & 1u);   // MMAs of k-tile i - USTAGES are done
        const uint8_t* rw = umma_smem + (i % NRAW) * (ra + rb);
        la.convert(rw, st, st + pa, g.relu_a);
        lb.convert(rw + ra, st + 2 * pa, st + 2 * pa + pb, g.relu_b);
        if (i + NRAW - 1 < nk) {        // refill the raw stage this thread emptied in the previous iteration
            const int t = i + NRAW - 1;
            const int64_t k0 = kbeg + (int64_t)t * UBK;
            const uint32_t dst = raw_base + (t % NRAW) * (ra + rb);
            la.issue(dst, t, k0, kend);
            lb.issue(dst + ra, t, k0, kend);
        }
        cp_async_commit();
        tc05::fence_smem_to_mma();
        tc05::fence_before();           // orders the drain's tcgen05.ld before the next MMA
        __syncthreads();
        const bool chunk_end = (i % UCH == UCH - 1) || (i == nk - 1);
        if (tid == 0) {
            tc05::fence_after();
            const uint32_t sa = tc05::smem_u32(st), sb = tc05::smem_u32(st + 2 * pa);
#pragma unroll
            for (int ks = 0; ks < UBK / 8; ++ks) {
                const uint64_t ah = tc05::make_desc(sa + ks * 2 * a_lbo, a_lbo, USBO), al = tc05::make_desc(sa + pa + ks * 2 * a_lbo, a_lbo, USBO);
                const uint64_t bh = tc05::make_desc(sb + ks * 2 * b_lbo, b_lbo, USBO), bl = tc05::make_desc(sb + pb + ks * 2 * b_lbo, b_lbo, USBO);
                tc05::mma_ss(tmem_d, al, bh, idesc, ((i % UCH) | ks) ? 1u : 0u);      // a chunk starts a fresh sum
                tc05::mma_ss(tmem_d, ah, bl, idesc, 1u);
                tc05::mma_ss(tmem_d, ah, bh, idesc, 1u);
            }
            tc05::commit(&empty_bar[s]);
            if (chunk_end) tc05::commit(&chunk_bar);
        }
        if (chunk_end) {
            // the chunk's MMAs are complete: warp w may read TMEM lanes 32 w .. 32 w + 31 = its output rows
            tc05::mbar_wait(&chunk_bar, chunk_phase);
            chunk_phase ^= 1u;
            __syncwarp();
            tc05::fence_after();
            if (MULTI && i != nk - 1) {             // drain: acc += TMEM tile (rounded fp32 adds)
#pragma unroll
                for (int cc = 0; cc < NACC / 32; ++cc) {
                    const int c0 = (2 * cc + chalf) * 16;
                    if (c0 < bn) {
                        uint32_t v[16];
                        tc05::ld16(tmem_d + ((uint32_t)lanes0 << 16) + (uint32_t)c0, v);
                        tc05::wait_ld();
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc[MULTI ? cc * 16 + j : 0] += __uint_as_float(v[j]);
                    }
                }
            }
        }
    }

    // epilogue, step 1: (registers +) TMEM -> row-major fp32 tile in the now idle operand stages (row stride bn + 4)
    cp_async_wait<0>();
    float* tile = reinterpret_cast<float*>(umma_smem);
    const int ts = bn + 4;
    {
        const int row = lanes0 + lane;
#pragma unroll
        for (int cc = 0; cc < (NACC >= 32 ? NACC / 32 : 1); ++cc) {
            const int c0 = (2 * cc + chalf) * 16;
            if (c0 < bn) {
                uint32_t u[16];
                tc05::ld16(tmem_d + ((uint32_t)lanes0 << 16) + (uint32_t)c0, u);
                tc05::wait_ld();
                float v[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(u[j]);
                if (MULTI) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] += acc[MULTI ? cc * 16 + j : 0];
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4*>(tile + row * ts + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            }
        }
    }
    tc05::fence_before();
    __syncthreads();
    if (warp == 0) tc05::tmem_free(tmem_d, NACC);

    // step 2: tile -> global, one row per warp pass with the lanes along the columns (coalesced); bias / residual /
    // relu / mask are applied here
    const bool first = (blockIdx.z == 0);
    const int64_t col = n0 + 4 * lane;
    const bool lane_on = 4 * lane < bn && col < g.N;
    const bool v4 = vec_c4 && col + 3 < g.N;
    float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane_on && v4 && first && g.bias) bias4 = *reinterpret_cast<const float4*>(g.bias + col);
    if (!vec_c4) {
        // rows that are not 16-byte aligned (N = intent_num = 1071 is odd): lanes on consecutive columns, scalar but
        // coalesced stores; everything that does not depend on the row (column guards, bias) is fetched once per lane
        float bj[NACC / 32 > 0 ? NACC / 32 : 1];
        bool on[NACC / 32 > 0 ? NACC / 32 : 1];
#pragma unroll
        for (int j = 0; j < (NACC / 32 > 0 ? NACC / 32 : 1); ++j) {
            const int c = lane + 32 * j;
            on[j] = c < bn && n0 + c < g.N;
            bj[j] = (on[j] && first && g.bias) ? g.bias[n0 + c] : 0.f;
        }
        const bool plain = g.accumulate == 0 && !g.mask && !(first && g.add);
        for (int r = warp; r < UM; r += UTHREADS / 32) {
            const int64_t gm = m0 + r;
            if (gm >= g.M) break;
            float* crow = g.C + gm * g.ldc + n0;
#pragma unroll
            for (int j = 0; j < (NACC / 32 > 0 ? NACC / 32 : 1); ++j) {
                if (!on[j]) continue;
                const int c = lane + 32 * j;
                float v = tile[r * ts + c] + bj[j];
                if (plain) {
                    crow[c] = g.relu_out ? fmaxf(v, 0.f) : v;
                    continue;
                }
                if (first && g.add) v += g.add[gm * g.ldadd + n0 + c];
                if (g.relu_out) v = fmaxf(v, 0.f);
                if (g.mask) v = (g.mask[gm * g.ldmask + n0 + c] > 0.f) ? v : 0.f;
                if (g.accumulate == 0) crow[c] = v;
                else if (g.accumulate == 1) crow[c] += v;
                else atomicAdd(crow + c, v);
            }
        }
        return;
    }
#pragma unroll 2
    for (int r = warp; r < UM; r += UTHREADS / 32) {
        const int64_t gm = m0 + r;
        if (gm >= g.M) break;
        if (!lane_on) continue;
        float4 v = *reinterpret_cast<const float4*>(tile + r * ts + 4 * lane);
        if (v4) {
            if (first) {
                v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
                if (g.add) {
                    const float4 a = *reinterpret_cast<const float4*>(g.add + gm * g.ldadd + col);
                    v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
                }
            }
            if (g.relu_out) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            if (g.mask) {
                const float4 m = *reinterpret_cast<const float4*>(g.mask + gm * g.ldmask + col);
                v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f; v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
            }
            float* c = g.C + gm * g.ldc + col;
            if (g.accumulate == 0) *reinterpret_cast<float4*>(c) = v;
            else if (g.accumulate == 1) {
                const float4 o = *reinterpret_cast<const float4*>(c);
                *reinterpret_cast<float4*>(c) = make_float4(o.x + v.x, o.y + v.y, o.z + v.z, o.w + v.w);
            } else {
                atomicAdd(c, v.x); atomicAdd(c + 1, v.y); atomicAdd(c + 2, v.z); atomicAdd(c + 3, v.w);
            }
        } else {
            gemm_store(g, gm, col, v.x, first);
            gemm_store(g, gm, col + 1, v.y, first);
            gemm_store(g, gm, col + 2, v.z, first);
            gemm_store(g, gm, col + 3, v.w, first);
        }
    }
}

}  // namespace umma
}  // namespace intel
#endif  // INTEL_EMU
