// mbarrier / bulk-copy (TMA) / elect wrappers shared by the kernels that stage data with cp.async.bulk
// (lec_score_mma.cu: label blobs; lec_featnet.cu: gathered feature rows).  sm_100a only.
#pragma once
#include "lec_common.cuh"

namespace lec {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Back-off of a warp that keeps finding an mbarrier phase incomplete: a waiting warp must not eat the issue slots of
// the working ones.
constexpr unsigned kMbarSleepNs = 32;
// Spins on the phase; a lost arrival traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned ok = 0;
    for (unsigned spin = 0; !ok; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok) {
            if (spin > 4) __nanosleep(kMbarSleepNs);
            if (spin > (1u << 22)) __trap();
        }
    }
}
// one non-blocking look at the phase
__device__ __forceinline__ bool mbar_test(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// one lane of the (converged) warp; the compiler knows the region under it runs on a single thread (ELECT), so operands
// of the uniform-datapath instructions inside (UTCHMMA, UTCBAR, UBLKCP) need no per-lane serialisation loop
__device__ __forceinline__ bool elect_one() {
    unsigned pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "@px mov.s32 %0, 1;\n\t}"
        : "+r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

}  // namespace lec
