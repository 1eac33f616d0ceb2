// HardNet 8x8 head on tensor cores: conv8x8(128->128, no bias) == GEMM [n, 8192] x [8192, 128], then BatchNorm and
// L2 normalisation (HardNet.py:86-101, 12-19).  A = trunk features in the L_HEAD layout written by the last conv layer
// ([patch/128][k/8][patch%128][8] fp16: 128 patches are the M rows of one tile), B = head weights [k/8][cout][8] fp16.
// One CTA per 128-patch tile streams K in 64-wide stages (A 16 KiB + B 16 KiB per stage, bulk copies, 6-stage ring),
// accumulates 128x128 fp32 in TMEM, and the epilogue thread of each row does BN + sum of squares + scale in registers.
#pragma once
#include "tcgen05.cuh"

namespace ag {
namespace tc {

constexpr int HEAD_K = 8192, HEAD_N = 128, HEAD_KS = 64, HEAD_STAGES = 6;
constexpr uint32_t HEAD_STAGE_A = (HEAD_KS / 8) * 128 * 16, HEAD_STAGE_B = (HEAD_KS / 8) * HEAD_N * 16;
constexpr size_t HEAD_SMEM = 1024 + (size_t)HEAD_STAGES * (HEAD_STAGE_A + HEAD_STAGE_B);

template <int BF>
__global__ void __launch_bounds__(192, 1) tc_head_kernel(const __half* __restrict__ feat, const __half* __restrict__ wh,
                                                          const float* __restrict__ bn /*scale[128], shift[128]*/, float* __restrict__ out,
                                                          int n, int group, const int* __restrict__ count) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty = full + HEAD_STAGES;
    uint64_t* done = empty + HEAD_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    unsigned char* sA = smem + 1024;
    unsigned char* sB = sA + (size_t)HEAD_STAGES * HEAD_STAGE_A;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;
    constexpr int NK = HEAD_K / HEAD_KS;  // 128 stages

    if (threadIdx.x == 0) {
        for (int s = 0; s < HEAD_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(128));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            const unsigned char* ga = reinterpret_cast<const unsigned char*>(feat) + (size_t)tile * (HEAD_K / 8) * 128 * 16;
            const unsigned char* gb = reinterpret_cast<const unsigned char*>(wh);
            for (int k = 0; k < NK; k++) {
                const int s = k % HEAD_STAGES;
                mbar_wait(&empty[s], ((k / HEAD_STAGES) & 1) ^ 1);
                mbar_expect_tx(&full[s], HEAD_STAGE_A + HEAD_STAGE_B);
                bulk_g2s(sA + (size_t)s * HEAD_STAGE_A, ga + (size_t)k * HEAD_STAGE_A, HEAD_STAGE_A, &full[s]);
                bulk_g2s(sB + (size_t)s * HEAD_STAGE_B, gb + (size_t)k * HEAD_STAGE_B, HEAD_STAGE_B, &full[s]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = (BF ? ((1u << 7) | (1u << 10)) : 0u) | (1u << 4) | ((uint32_t)(HEAD_N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // BF: bf16 operands
            for (int k = 0; k < NK; k++) {
                const int s = k % HEAD_STAGES;
                mbar_wait(&full[s], (k / HEAD_STAGES) & 1);
                tc_fence_after();
                const uint32_t a0 = smem_u32(sA + (size_t)s * HEAD_STAGE_A), b0 = smem_u32(sB + (size_t)s * HEAD_STAGE_B);
#pragma unroll
                for (int j = 0; j < HEAD_KS / 16; j++) {
                    const uint64_t da = make_desc(a0 + (uint32_t)(2 * j) * 128u * 16u, 128u * 16u, 128u);
                    const uint64_t db = make_desc(b0 + (uint32_t)(2 * j) * HEAD_N * 16u, HEAD_N * 16u, 128u);
                    umma_f16(tmem, da, db, idesc, (k | j) != 0);
                }
                umma_commit(&empty[s]);
            }
            umma_commit(done);
        }
    } else {
        const int q = warp & 3;
        mbar_wait(done, 0);
        tc_fence_after();
        const int pi = tile * 128 + q * 32 + lane;
        const bool ok = pi < n && (count == nullptr || (pi % group) < count[pi / group]);
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
        float ss = 0.f;
        // pass 1: sum of squares of the BatchNorm-ed row; pass 2: reload, scale, store (keeps registers low)
#pragma unroll 1
        for (int c0 = 0; c0 < HEAD_N; c0 += 32) {
            uint32_t r[32];
            tmem_ld32(taddr + c0, r);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; e++) {
                const float v = fmaf(__uint_as_float(r[e]), __ldg(bn + c0 + e), __ldg(bn + 128 + c0 + e));
                ss = fmaf(v, v, ss);
            }
        }
        const float inv = 1.0f / sqrtf(ss + 1e-8f);
#pragma unroll 1
        for (int c0 = 0; c0 < HEAD_N; c0 += 32) {
            uint32_t r[32];
            tmem_ld32(taddr + c0, r);
            tmem_ld_wait();
            if (ok) {
                float4* o = reinterpret_cast<float4*>(out + (size_t)pi * 128 + c0);
#pragma unroll
                for (int e = 0; e < 32; e += 4) {
                    float4 v;
                    v.x = fmaf(__uint_as_float(r[e + 0]), __ldg(bn + c0 + e + 0), __ldg(bn + 128 + c0 + e + 0)) * inv;
                    v.y = fmaf(__uint_as_float(r[e + 1]), __ldg(bn + c0 + e + 1), __ldg(bn + 128 + c0 + e + 1)) * inv;
                    v.z = fmaf(__uint_as_float(r[e + 2]), __ldg(bn + c0 + e + 2), __ldg(bn + 128 + c0 + e + 2)) * inv;
                    v.w = fmaf(__uint_as_float(r[e + 3]), __ldg(bn + c0 + e + 3), __ldg(bn + 128 + c0 + e + 3)) * inv;
                    o[e / 4] = v;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128));
    }
}

// ---- AffNet / OriNet heads on tensor cores -------------------------------------------------------------------------------
// conv8x8(64 -> 3) resp. the padded conv8x8(64 -> 2) seen as 18 shifted dot products (nets_simt.cu) == GEMM [n, 4096] x
// [4096, 32] with fp32-grade operands: the last conv layer writes its output as fp16 hi + lo planes in the L_HEAD layout, the head
// weights are stored as [k/8][W_hi rows 0..31 | W_lo rows 32..63][8], and per K step the issuer runs A_hi x [W_hi ; W_lo]
// (N = 64) and A_lo x W_hi (N = 32); the epilogue adds the two accumulator halves and applies the reference's post-processing
// (architectures.py:57-59,76-82,228-230; LAF.py:276-291).  One CTA per 128-patch tile, K streamed in 64-wide stages.
// The tensor core adds into its fp32 accumulator with truncation, and the error grows with the length of the running sum (measured:
// one accumulator over all 512 MMAs costs 2.3e-4 rad of OriNet angle against 2.6e-5 with an fp32 FMA chain).  The K stages
// therefore rotate over HX_G = 8 accumulator column groups (all 512 TMEM columns) and the epilogue adds the groups in fp32.
constexpr int HX_K = 4096, HX_NP = 32, HX_KS = 64, HX_STAGES = 5, HX_G = 8;
constexpr uint32_t HX_STAGE_A = (HX_KS / 8) * 128 * 16, HX_STAGE_B = (HX_KS / 8) * (2 * HX_NP) * 16;
constexpr size_t HX_SMEM = 1024 + (size_t)HX_STAGES * (2 * HX_STAGE_A + HX_STAGE_B);
constexpr size_t HX_PLANE_TILE = (size_t)(HX_K / 8) * 128 * 16;   // bytes of one 128-patch tile in one plane

template <int KIND /* 0 AffNet, 1 OriNet */>
__global__ void __launch_bounds__(192, 1) tc_headx_kernel(const __half* __restrict__ feat, const __half* __restrict__ wh, const float* __restrict__ bias,
                                                           const float inv_scale, float* __restrict__ out, float* __restrict__ angle_out, float* __restrict__ raw_out, int n, int group,
                                                           const int* __restrict__ count) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty = full + HX_STAGES;
    uint64_t* done = empty + HX_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    unsigned char* sA = smem + 1024;                                    // [stage][hi | lo]
    unsigned char* sB = sA + (size_t)HX_STAGES * 2 * HX_STAGE_A;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x, tiles = gridDim.x;
    constexpr int NK = HX_K / HX_KS;

    {   // a tile without a single live patch has nothing to do (rows beyond count[] of every image it touches)
        int live = 0;
        if (threadIdx.x < 128) {
            const int pi = tile * 128 + threadIdx.x;
            live = pi < n && (count == nullptr || (pi % group) < count[pi / group]);
        }
        if (!__syncthreads_or(live)) return;
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < HX_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(HX_G * 2 * HX_NP));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            const unsigned char* ga = reinterpret_cast<const unsigned char*>(feat) + (size_t)tile * HX_PLANE_TILE;
            const unsigned char* gl = ga + (size_t)tiles * HX_PLANE_TILE;
            const unsigned char* gb = reinterpret_cast<const unsigned char*>(wh);
            for (int k = 0; k < NK; k++) {
                const int s = k % HX_STAGES;
                mbar_wait(&empty[s], ((k / HX_STAGES) & 1) ^ 1);
                mbar_expect_tx(&full[s], 2 * HX_STAGE_A + HX_STAGE_B);
                bulk_g2s(sA + (size_t)s * 2 * HX_STAGE_A, ga + (size_t)k * HX_STAGE_A, HX_STAGE_A, &full[s]);
                bulk_g2s(sA + (size_t)s * 2 * HX_STAGE_A + HX_STAGE_A, gl + (size_t)k * HX_STAGE_A, HX_STAGE_A, &full[s]);
                bulk_g2s(sB + (size_t)s * HX_STAGE_B, gb + (size_t)k * HX_STAGE_B, HX_STAGE_B, &full[s]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_st = (1u << 4) | ((uint32_t)((2 * HX_NP) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            constexpr uint32_t idesc_hi = (1u << 4) | ((uint32_t)(HX_NP >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            for (int k = 0; k < NK; k++) {
                const int s = k % HX_STAGES;
                mbar_wait(&full[s], (k / HX_STAGES) & 1);
                tc_fence_after();
                const uint32_t a0 = smem_u32(sA + (size_t)s * 2 * HX_STAGE_A), b0 = smem_u32(sB + (size_t)s * HX_STAGE_B);
#pragma unroll
                for (int j = 0; j < HX_KS / 16; j++) {
                    const uint64_t da = make_desc(a0 + (uint32_t)(2 * j) * 128u * 16u, 128u * 16u, 128u);
                    const uint64_t dl = make_desc(a0 + HX_STAGE_A + (uint32_t)(2 * j) * 128u * 16u, 128u * 16u, 128u);
                    const uint64_t db = make_desc(b0 + (uint32_t)(2 * j) * (2 * HX_NP) * 16u, (2 * HX_NP) * 16u, 128u);
                    const uint32_t d = tmem + (uint32_t)((k % HX_G) * 2 * HX_NP);
                    umma_f16(d, da, db, idesc_st, (k >= HX_G) || j != 0);   // A_hi x [W_hi ; W_lo]
                    umma_f16(d, dl, db, idesc_hi, 1);                        // A_lo x W_hi -> hi columns
                }
                umma_commit(&empty[s]);
            }
            umma_commit(done);
        }
    } else {
        const int q = warp & 3;
        mbar_wait(done, 0);
        tc_fence_after();
        const int pi = tile * 128 + q * 32 + lane;
        const bool ok = pi < n && (count == nullptr || (pi % group) < count[pi / group]);
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
        constexpr int NO = KIND == 0 ? 3 : 18;
        float acc[NO];
#pragma unroll
        for (int o = 0; o < NO; o++) acc[o] = 0.f;
#pragma unroll 1
        for (int g = 0; g < HX_G; g++) {
            uint32_t r[32], r2[32];
            tmem_ld32(taddr + g * 2 * HX_NP, r);
            tmem_ld32(taddr + g * 2 * HX_NP + HX_NP, r2);
            tmem_ld_wait();
#pragma unroll
            for (int o = 0; o < NO; o++) acc[o] += __uint_as_float(r[o]) + __uint_as_float(r2[o]);
        }
        if (ok) {
            if (KIND == 0) {
                const float s0 = acc[0] * inv_scale, s1 = acc[1] * inv_scale, s2 = acc[2 % NO] * inv_scale;
                const float a00 = 1.0f + tanhf(s0 + bias[0]), a01 = 0.f, a10 = tanhf(s1 + bias[1]), a11 = 1.0f + tanhf(s2 + bias[2]);
                if (raw_out) { raw_out[(size_t)pi * 3] = a00; raw_out[(size_t)pi * 3 + 1] = a10; raw_out[(size_t)pi * 3 + 2] = a11; }   // convertJIT/AffNetJIT.pt: xy + [1, 0, 1]
                if (out) {
                    const float det = sqrtf(fabsf(a00 * a11 - a10 * a01 + 1e-10f));
                    const float b2a2 = sqrtf(a01 * a01 + a00 * a00);
                    float* o = out + (size_t)pi * 4;
                    o[0] = b2a2 / det; o[1] = 0.f;
                    o[2] = (a11 * a01 + a10 * a00) / (b2a2 * det); o[3] = det / b2a2;
                }
            } else {
                float m0 = 0.f, m1 = 0.f;
#pragma unroll
                for (int o = 0; o < 9; o++) {
                    m0 += tanhf(acc[o % NO] * inv_scale + bias[0]);
                    m1 += tanhf(acc[(9 + o) % NO] * inv_scale + bias[1]);
                }
                m0 /= 9.0f; m1 /= 9.0f;
                if (raw_out) { raw_out[(size_t)pi * 2] = m0; raw_out[(size_t)pi * 2 + 1] = m1; }   // convertJIT/OriNetJIT.pt: the mean of tanh over the 3x3 map
                const float ang = atan2f(m0 + 1e-8f, m1 + 1e-8f);
                if (angle_out) angle_out[pi] = ang;
                if (out) {
                    const float c = cosf(ang), sn = sinf(ang);
                    float* o = out + (size_t)pi * 4;
                    o[0] = c; o[1] = sn; o[2] = -sn; o[3] = c;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(HX_G * 2 * HX_NP));
    }
}

}  // namespace tc
}  // namespace ag
