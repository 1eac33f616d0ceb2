// tcgen05 building blocks shared by the tensor-core kernels (tcx_first.cuh, tcx_conv.cuh, tc_head.cuh), sm_100a: PTX wrappers
// for mbarriers, bulk copies, UMMA descriptors and MMAs, TMEM loads and fences, and the source description of the fused first layer.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace ag {
namespace tc {

// Developer-only role profiler (build with AG_XPROF=1, scripts/role_prof_x.py): cycles a warp role spends in its loop and waiting on
// each of its barriers.  Compiled out of the product library.
#ifdef AG_ROLE_PROF
#define RP_DECL unsigned long long rp_t0 = clock64(), rp_w[4] = {0, 0, 0, 0}
#define RP_WAIT(i, stmt) do { const unsigned long long rp_t = clock64(); stmt; rp_w[i] += clock64() - rp_t; } while (0)
#else
#define RP_DECL
#define RP_WAIT(i, stmt) stmt
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// no-swizzle K-major UMMA shared-memory descriptor (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// AG_MBAR_HINT_NS > 0: try_wait carries a suspend-time hint, so a waiting warp sleeps in hardware until the phase completes (or the hint
// expires) instead of re-issuing try_wait + branch every ~40 clk (ncu source view without the hint: the polling loops were 7.6 % of
// tcx_first_kernel's and 16 % of a tcx_conv_kernel's issued instructions; step time -0.5 .. 1 %)
#ifndef AG_MBAR_HINT_NS
#define AG_MBAR_HINT_NS 200000
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#if AG_MBAR_HINT_NS > 0
    asm volatile(
        "{\n .reg .pred P;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 P, [%0], %1, %2;\n @P bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n" ::"r"(smem_u32(bar)),
        "r"(parity), "r"((uint32_t)AG_MBAR_HINT_NS)
        : "memory");
#else
    asm volatile(
        "{\n .reg .pred P;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 P, [%0], %1;\n @P bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
#endif
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(adesc),
                 "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
// Descriptor-lo form: the hi word of every no-swizzle descriptor here is the constant 0x4008 (SBO = 128 B, version 1), so the
// issuer only does one integer add per operand.  ACC is a compile-time accumulate flag.
constexpr uint32_t DESC_HI = 0x4008u;
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr >> 4) & 0x3FFFu) | ((lbo_bytes >> 4) << 16); }
template <int ACC>
__device__ __forceinline__ void umma_f16_lo(uint32_t tmem_d, uint32_t alo, uint32_t blo, uint32_t idesc) {
    asm volatile(
        "{\n .reg .pred p;\n .reg .b64 da, db;\n setp.ne.u32 p, %4, 0;\n mov.b64 da, {%1, %5};\n mov.b64 db, {%2, %5};\n"
        " tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n}\n" ::"r"(tmem_d),
        "r"(alo), "r"(blo), "r"(idesc), "n"(ACC), "r"(DESC_HI)
        : "memory");
}
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n .reg .pred P;\n elect.sync _|P, 0xffffffff;\n selp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Source of the first kernel (tcx_first.cuh): either materialised patches [n,32,32] fp32, or the pyramid + keypoints
// (the affine bilinear sampler of LAF.py:313-372 runs inside the kernel; patches never touch HBM).
struct PyrGeomTC {
    int n_octaves, n_levels;
    int h[AG_MAX_OCTAVES], w[AG_MAX_OCTAVES];
    long long off[AG_MAX_OCTAVES][AG_MAX_LEVELS];
};
struct FirstSrc {
    const float* patches;   // if non-NULL: [n][32][32]
    const float* pyr;       // else: pyramid base, rows (b, i) = (pi / cap, pi % cap)
    const float* lafs;      // [B*cap][2][3] normalised
    const int* oct;
    const int* lvl;
    int cap;
    const float* w1;        // [9][C1] fp32 (BatchNorm folded)
    float w1_scale, w1_inv; // tensor-core layer 1: weights are used times w1_scale (a power of two), accumulators times w1_inv
    const float* b1;        // [C1]
    PyrGeomTC geom;
};

}  // namespace tc
}  // namespace ag
