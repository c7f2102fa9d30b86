// tc05.cuh -- thin PTX wrappers for the sm_100a tensor-core path (tcgen05.mma kind::i8, TMEM, mbarriers) used by the
// bit-plane kernels (planes.cu) and the microbenchmarks under profiles/microbench.  Encodings follow
// cute/arch/mma_sm100_desc.hpp (UMMA::SmemDescriptor, UMMA::InstrDescriptor).
#pragma once
#include <cstdint>

namespace tc05 {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Shared-memory matrix descriptor, SWIZZLE_NONE ("interleaved"): core matrices of 8 rows x 16 bytes (128 contiguous bytes).
//   K-major operand : rows = M/N index, 16 bytes = 16 K elements; lbo = bytes between core matrices adjacent in K,
//                     sbo = bytes between core matrices adjacent in M/N.
//   MN-major operand: rows = K index, 16 bytes = 16 M/N elements; lbo = bytes between groups of 8 K rows,
//                     sbo = bytes between 16-element units along M/N.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;  // descriptor version 1 (Blackwell); base offset 0; layout type 0 = no swizzle
    return d;
}

// Instruction descriptor for kind::i8: D = S32, A = B = signed 8-bit; a_mn / b_mn: operand is MN-major
__host__ __device__ constexpr uint32_t instr_desc_i8(uint32_t M, uint32_t N, bool a_mn, bool b_mn) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}

// The same MMA from the LOW descriptor words (address | leading byte offset); the high words (stride byte offset, descriptor
// version) are compile-time immediates, so consecutive descriptors differ by one 32-bit add.
template <uint32_t HI_A, uint32_t HI_B>
__device__ __forceinline__ void mma_i8_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %6};\n\tmov.b64 db, {%2, %7};\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(0u), "n"(HI_A), "n"(HI_B)
        : "memory");
}

// One lane of a converged warp (elect.sync).  The tcgen05 issue loops run warp-uniformly and predicate only the tensor-core
// instructions with this: inside `if (lane == 0)` the compiler cannot keep the operands in uniform registers and wraps every
// UTCIMMA in an ELECT / R2UR.BROADCAST loop (measured: 155-240 instructions per stage instead of ~25).
__device__ __forceinline__ bool elect_one(uint32_t &leader) {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred px;\n\t"
        "elect.sync %1|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}\n"
        : "=r"(pred), "=r"(leader));
    return pred != 0;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t leader;
    return elect_one(leader);
}

// arrives (count 1) on the mbarrier once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}\n" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "TC05_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TC05_DONE_%=;\n\t"
        "bra TC05_WAIT_%=;\n\t"
        "TC05_DONE_%=:\n\t}\n" ::"r"(mbar),
        "r"(parity)
        : "memory");
}

// tight poll (test_wait never suspends): for the one thread whose reaction time paces the tensor pipe
__device__ __forceinline__ void mbar_spin(uint32_t mbar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done)
                     : "r"(mbar), "r"(parity)
                     : "memory");
}

// Bulk asynchronous copy global -> shared (the TMA engine's 1-D form): `bytes` (multiple of 16, both addresses 16-byte aligned)
// land in shared memory and are counted as completed transaction bytes on `mbar`, which must expect them (mbar_expect_tx).
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_saddr, const void *src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_saddr), "l"(src), "r"(bytes),
                 "r"(mbar)
                 : "memory");
}

// long waits (an epilogue waiting for a whole CTA's worth of MMAs): back off so the spinning warps leave the issue slots alone
__device__ __forceinline__ void mbar_wait_sleep(uint32_t mbar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(mbar), "r"(parity)
            : "memory");
        if (!done) __nanosleep(500);
    }
}

// generic-proxy shared-memory writes -> visible to the tensor core (async proxy)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc_512(uint32_t slot_saddr) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(slot_saddr) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}

// 16 consecutive TMEM columns of this thread's lane (warp w of the CTA's first four reads lanes 32 w .. 32 w + 31)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 bits -> 32 bytes of 0/1 (byte i = bit i): four bits at a time, (nibble * 0x00204081) & 0x01010101
__device__ __forceinline__ void expand_bits32(uint32_t w, uint4 &lo, uint4 &hi) {
    lo.x = ((w & 0xFu) * 0x00204081u) & 0x01010101u;
    lo.y = (((w >> 4) & 0xFu) * 0x00204081u) & 0x01010101u;
    lo.z = (((w >> 8) & 0xFu) * 0x00204081u) & 0x01010101u;
    lo.w = (((w >> 12) & 0xFu) * 0x00204081u) & 0x01010101u;
    hi.x = (((w >> 16) & 0xFu) * 0x00204081u) & 0x01010101u;
    hi.y = (((w >> 20) & 0xFu) * 0x00204081u) & 0x01010101u;
    hi.z = (((w >> 24) & 0xFu) * 0x00204081u) & 0x01010101u;
    hi.w = ((w >> 28) * 0x00204081u) & 0x01010101u;
}

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void st_shared_v4(uint32_t saddr, const uint4 &v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

}  // namespace tc05
