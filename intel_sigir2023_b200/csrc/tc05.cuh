// tcgen05 / tensor-memory primitives shared by the tcgen05 kernels (trunk_tc.cu, gru_tc.cu, the GEMMs).  Every form used here was
// checked bit-exact on a B200 with tests/hw/umma_probe.cu (profiles/r02_probe.md):
//   * kind::tf32 MMA with the A operand in shared memory (SS) or in tensor memory (TS), fp32 accumulator in TMEM;
//   * the disable-output-lane mask (four 32-bit words, bit set = accumulator lane not written): two sessions that share
//     a 128-row tile multiply against their own B operand without spending accumulator columns on the other's;
//   * K-major no-swizzle operands as "quad-slab" planes [k / 4][row][4] (LBO = rows * 16, SBO = 128);
//   * MN-major operands (the contraction runs over the tile ROWS) from natural [row][32 floats] tiles whose 32-byte
//     chunk index is XORed with (row & 3): SWIZZLE_128B_BASE32B, LBO = stride between 32-column groups, SBO = 512.
#pragma once
#ifndef INTEL_EMU
#include <stdint.h>

namespace intel {
namespace tc05 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "TC05_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra TC05_DONE;\n"
        "bra TC05_WAIT;\n"
        "TC05_DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp (the MMA operands then stay in uniform registers instead of going through R2UR per MMA)
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(p));
    return p != 0;
}
// one arrival on the mbarrier once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the tensor core (async proxy)
__device__ __forceinline__ void fence_smem_to_mma() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// shared-memory matrix descriptor; layout: 0 = no swizzle, 1 = SWIZZLE_128B_BASE32B, 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout = 0) {
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;                          // descriptor version of sm_100
    d |= (uint64_t)layout << 61;
    return d;
}
// instruction descriptor: D = f32, A = B = tf32, a_mn / b_mn = 1 for an MN-major operand
__device__ __forceinline__ uint32_t make_idesc(int M, int N, int a_mn = 0, int b_mn = 0) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

struct LaneMask { uint32_t w[4]; };     // bit set = lane disabled
__device__ __forceinline__ LaneMask mask_rows(int first, int count) {       // enable lanes [first, first + count), multiples of 32
    LaneMask m;
#pragma unroll
    for (int i = 0; i < 4; ++i) m.w[i] = (32 * i >= first && 32 * i < first + count) ? 0u : 0xffffffffu;
    return m;
}

__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(d), "l"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc, const LaneMask& m) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n}" ::"r"(d),
                 "l"(a), "l"(b), "r"(idesc), "r"(acc), "r"(m.w[0]), "r"(m.w[1]), "r"(m.w[2]), "r"(m.w[3])
                 : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}" ::"r"(d), "r"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc, const LaneMask& m) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n}" ::"r"(d),
                 "r"(a), "l"(b), "r"(idesc), "r"(acc), "r"(m.w[0]), "r"(m.w[1]), "r"(m.w[2]), "r"(m.w[3])
                 : "memory");
}

// tensor memory <-> registers: the calling warp's 32 lanes, 32 consecutive columns, one row per thread.
// ld32 does NOT wait: call wait_ld() before the registers are read.  ld8 / st8 (the parked weight-gradient and dQ | dK | dV
// tiles of trunk_bwd_kernel) are covered by the GPU parity tests of that kernel rather than by the probe.
__device__ __forceinline__ void ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
        "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr), "r"(r[0]),
        "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]),
        "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {       // one warp; cols: power of two >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

}  // namespace tc05
}  // namespace intel
#endif  // INTEL_EMU
