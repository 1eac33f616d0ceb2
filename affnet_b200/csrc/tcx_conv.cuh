// Second-generation tensor-core (tcgen05) 3x3 convolution engine (sm_100a): row tiles without x padding, taps of one kernel row
// stacked along N.
//
// Measured on B200 (tests/probe/tc_rates.cu): one tcgen05.mma kind::f16 (M = 128, K = 16) costs max(47.5, N/2) clk whatever its
// operands' source, so an MMA with N = 16 .. 64 leaves 66 - 90 % of the tensor pipe idle.  The first-generation engine (tc_conv.cuh)
// issued one MMA per tap (N = 16 .. 64); here the three taps of a kernel ROW share one MMA:
//
//   pixel planes are stored WITHOUT x padding, so that an M = 128 tile is 128 consecutive pixels = whole image rows (4 rows of 32,
//   8 rows of 16, or 8 rows of 8 of TWO patches interleaved row by row), and every warp of the epilogue owns whole rows;
//   for kernel row dy the A operand is the input plane advanced by dy rows (descriptor start address; a zero row above and below
//   the plane in shared memory gives the y padding) and the B operand stacks the three taps of that row along N:
//        D[q, (dx, c)] += sum_ci  in[q + (dy-1) W, ci] * w[dy][dx][ci][c]             one MMA per (dy, 16 input channels), N = 3 C
//   the x shift moves to the epilogue:   out[p, c] = D[p-1, (0,c)] + D[p, (1,c)] + D[p+1, (2,c)]   (warp shuffles inside an image
//   row; the neighbour outside the row is the zero padding).
// Stride-2 layers read four parity planes; the taps dx = 0 and dx = 2 share the odd-x plane (N = 2 C), dx = 1 reads the even-x
// plane (N = C):   out[x] = Dodd[x-1, dx0] + Dodd[x, dx2] + Deven[x, dx1].
// Split precision as before: x = hi + lo fp16 planes (SA), w = hi + lo fp16 copies (SW), D = A_hi W_hi + A_hi W_lo + A_lo W_hi, each
// product its own MMA into the SAME accumulator columns (at N >= 96 the MMAs are math bound, stacking hi | lo along N buys nothing).
//
// Activations between layers (HBM): fp16, 16-byte slots of 8 channels, [unit][channel group (hi groups, then lo groups)][plane][slot],
// data rows only (the consumer's loader places them between zero rows in shared memory):
//   L_S2_16  stride-2 consumer on a 32x32 map   unit = patch   4 parity planes x 256 slots  slot = (y/2)*16 + x/2, plane = (y&1)*2 + (x&1)
//   L_S1_16  stride-1 consumer on a 16x16 map   unit = patch   256 slots                    slot = y*16 + x
//   L_S2_8P  stride-2 consumer on a 16x16 map   unit = PAIR    4 parity planes x 128 slots  slot = ((y/2)*2 + p)*8 + x/2
//   L_S1_8P  stride-1 consumer on an 8x8 map    unit = PAIR    128 slots                    slot = (y*2 + p)*8 + x       (p = patch & 1)
//   L_HEAD   the 8x8 head GEMM's A operand (tc_head.cuh): [patch/128][pixel*C/8 + c/8][patch%128][8] (+ a residual plane behind it)
//
// Warp roles: 0 .. EW-1 epilogue (4 warps per set, EW/4 sets taking tiles in turn: one tcgen05.ld stream reads 43 B/clk per warp, so wide
// accumulators want more readers) | EW loader (cp.async.bulk per channel group and plane) | EW+1 MMA issuer (the highest warp id: the SMSP
// arbiter prefers it).
#pragma once
#include <cuda_bf16.h>

#include "tc_conv.cuh"

namespace ag {
namespace tcx {

using namespace ag::tc;

// Developer-only role profiler (scripts/role_prof_x.py, build with AG_XPROF=1): cycles of one warp of every role and its barrier waits.
#ifdef AG_ROLE_PROF
__device__ unsigned long long g_xprof[8][160][20];   // [slot: 0 tcx_first, l = conv layer l+1][CTA][role*5 + k]
#define XP_STORE(slot, role) do { if (lane == 0) { unsigned long long* d_ = g_xprof[slot][blockIdx.x + gridDim.x * blockIdx.y] + (role) * 5; \
    d_[0] = clock64() - rp_t0; d_[1] = rp_w[0]; d_[2] = rp_w[1]; d_[3] = rp_w[2]; d_[4] = rp_w[3]; } } while (0)
#else
#define XP_STORE(slot, role)
#endif

enum XLayout { L_S2_16 = 0, L_S1_16 = 1, L_S2_8P = 2, L_S1_8P = 3, L_HEAD = 4 };

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

// Cluster multicast (the two CTAs that split a layer's output channels read the SAME input unit): a bulk copy lands at the same
// shared-memory offset of every CTA in the mask and completes bytes on the mbarrier at the same offset of each; a commit arrives on the
// barrier at the same offset of each.
__device__ __forceinline__ void bulk_g2s_mc(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint16_t mask) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Operand type of an engine instance: BF = 0 fp16, BF = 1 bf16 (BASELINE.json configs[4]: "bf16 HardNet tensor-core path"); the MMA kind
// is kind::f16 for both, the instruction descriptor carries the A / B formats.
template <int BF> struct XFmt { static constexpr uint32_t IDESC = BF ? ((1u << 7) | (1u << 10)) : 0u; };
template <int BF>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    if (BF) { const __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<const uint32_t*>(&h); }
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
template <int BF>
__device__ __forceinline__ float2 unpack2(uint32_t u) {
    if (BF) return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
    return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
// 8 fp32 values -> 8 16-bit floats (hi) and, when LO, the residuals v - hi rounded to the same format; the residual is taken from the
// packed hi (one F2FP per pair)
template <int LO, int BF = 0>
__device__ __forceinline__ void split_pack8(const float* v, uint4& hi, uint4& lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        h[i] = pack2<BF>(v[2 * i], v[2 * i + 1]);
        if (LO) {
            const float2 f = unpack2<BF>(h[i]);
            l[i] = pack2<BF>(v[2 * i] - f.x, v[2 * i + 1] - f.y);
        } else l[i] = 0;
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// Byte residual planes (SA / OSA = 2): the fp16 residual rounded to its high byte (= e5m2).  Emulation (scripts/emu_residual_bits.py):
// AffNet's output moves by 5e-6 when the residual of an activation keeps 2 mantissa bits (budget 5e-5), so the planes that cross HBM
// in front of the bandwidth-bound stride-2 layers are stored at half the size and expanded in shared memory by the consumer.
__device__ __forceinline__ uint2 pack_lo8(const uint4& lo) {
    const uint32_t t0 = lo.x + 0x00800080u, t1 = lo.y + 0x00800080u, t2 = lo.z + 0x00800080u, t3 = lo.w + 0x00800080u;   // round the magnitude to 8 bits
    return make_uint2(__byte_perm(t0, t1, 0x7531), __byte_perm(t2, t3, 0x7531));
}

// slots per channel group and unit of an HBM activation layout, and patches per unit
__host__ __device__ constexpr int layout_slots(int lay) { return lay == L_S2_16 ? 1024 : lay == L_S1_16 ? 256 : lay == L_S2_8P ? 512 : 128; }
__host__ __device__ constexpr int layout_pair(int lay) { return (lay == L_S2_8P || lay == L_S1_8P) ? 1 : 0; }
// slot of pixel (y, x) of patch parity p in a layout
__host__ __device__ constexpr int layout_slot(int lay, int y, int x, int p) {
    return lay == L_S2_16 ? ((y & 1) * 2 + (x & 1)) * 256 + (y >> 1) * 16 + (x >> 1)
         : lay == L_S1_16 ? y * 16 + x
         : lay == L_S2_8P ? ((y & 1) * 2 + (x & 1)) * 128 + ((y >> 1) * 2 + p) * 8 + (x >> 1)
                          : (y * 2 + p) * 8 + x;
}

// Geometry of a layer's input in shared memory.  H: input map edge, STRIDE 1 | 2.
template <int H, int STRIDE>
struct XIn {
    static constexpr int HOUT = H / STRIDE;
    static constexpr int PAIR = (HOUT == 8) ? 1 : 0;              // two patches per tile, interleaved row by row
    static constexpr int W = HOUT;                                // pixels of one patch per image row
    static constexpr int RW = W * (1 + PAIR);                     // slots per (interleaved) row
    static constexpr int TILES = HOUT * RW / 128;                 // 8 | 2 | 1
    static constexpr int NPLANES = (STRIDE == 1) ? 1 : 4;
    static constexpr int DATA = HOUT * RW;                        // data slots per plane
    static constexpr int PLANE = DATA + RW;                       // + one zero row above
    static constexpr int SLOT_STAGE = NPLANES * PLANE;            // stride 1: the zero row BELOW a stage is the next stage's (or the group's trailing) zero row
    static constexpr int LAYOUT = (STRIDE == 2) ? (PAIR ? L_S2_8P : L_S2_16) : (PAIR ? L_S1_8P : L_S1_16);
    static_assert(HOUT == 8 || HOUT == 16 || HOUT == 32, "map sizes of the three nets");
    static_assert(!(STRIDE == 1 && H == 32), "the 32x32 stride-1 layer lives in tcx_first.cuh");
};

// MMAs of one stride-2 output tile (M = 128) into accumulator columns d .. d + 3 NT: for kernel row dy and 16 input channels the odd-x
// plane (taps dx = 0 | 2, N = 2 NT, columns d .. d + 2 NT) and the even-x plane (tap dx = 1, N = NT, columns d + 2 NT ..), each as the
// A_hi W_hi, A_hi W_lo (SW) and A_lo W_hi (SA) products.  a_t: the tile's first slot of the stage (16-byte units), PL / RW: plane and
// row slots, GS: slots per channel group; w_base: the layer's weight blocks (16-byte units).  Shared by tcx_conv_kernel and the fused
// layer 3 of tcx_first_kernel, so both issue the same MMAs in the same order.
template <int KC, int NT, int PL, int RW, int GS, int SA, int SW, int BF>
__device__ __forceinline__ void xmma_s2_tile(uint32_t d, uint32_t a_t, uint32_t w_base) {
    constexpr uint32_t idesc2 = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)((2 * NT) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr uint32_t idesc1 = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr int NRO = (1 + SW) * 2 * NT, NRE = (1 + SW) * NT;   // weight rows per K group: odd-x plane [hi: dx0 dx2][lo: ...], even-x plane [hi: dx1][lo: dx1]
    constexpr uint32_t LBO_A = ((uint32_t)GS) << 16;
#pragma unroll
    for (int dy = 0; dy < 3; dy++) {
        const int py = (dy == 1) ? 0 : 1, ro = (dy == 0) ? 0 : 1;
#pragma unroll
        for (int j = 0; j < KC / 2; j++) {
            const uint32_t blk = w_base + (uint32_t)((dy * (KC / 2) + j) * 2 * (NRO + NRE));
            const uint32_t bo_hi = (blk & 0x3FFFu) | ((uint32_t)NRO << 16), bo_lo = ((blk + 2 * NT) & 0x3FFFu) | ((uint32_t)NRO << 16);
            const uint32_t be = blk + 2 * NRO;
            const uint32_t be_hi = (be & 0x3FFFu) | ((uint32_t)NRE << 16), be_lo = ((be + NT) & 0x3FFFu) | ((uint32_t)NRE << 16);
            // odd-x plane (px = 1): taps dx = 0 and dx = 2
            const uint32_t ao = a_t + (uint32_t)((py * 2 + 1) * PL + ro * RW);
            const uint32_t ao_hi = ((ao + (uint32_t)(2 * j * GS)) & 0x3FFFu) | LBO_A, ao_lo = ((ao + (uint32_t)((KC + 2 * j) * GS)) & 0x3FFFu) | LBO_A;
            if (dy == 0 && j == 0) umma_f16_lo<0>(d, ao_hi, bo_hi, idesc2); else umma_f16_lo<1>(d, ao_hi, bo_hi, idesc2);
            if (SW) umma_f16_lo<1>(d, ao_hi, bo_lo, idesc2);
            if (SA) umma_f16_lo<1>(d, ao_lo, bo_hi, idesc2);
            // even-x plane (px = 0): tap dx = 1
            const uint32_t ae = a_t + (uint32_t)((py * 2 + 0) * PL + ro * RW);
            const uint32_t ae_hi = ((ae + (uint32_t)(2 * j * GS)) & 0x3FFFu) | LBO_A, ae_lo = ((ae + (uint32_t)((KC + 2 * j) * GS)) & 0x3FFFu) | LBO_A;
            const uint32_t de = d + (uint32_t)(2 * NT);
            if (dy == 0 && j == 0) umma_f16_lo<0>(de, ae_hi, be_hi, idesc1); else umma_f16_lo<1>(de, ae_hi, be_hi, idesc1);
            if (SW) umma_f16_lo<1>(de, ae_hi, be_lo, idesc1);
            if (SA) umma_f16_lo<1>(de, ae_lo, be_hi, idesc1);
        }
    }
}

struct XArgs {
    const __half* in;     // HBM activation buffer in the layer's input layout
    void* out;            // next layer's buffer
    const __half* wpk;    // packed weights (tcx_pack_layer)
    const float* bias;    // [COUT]
    float inv_scale;      // 1 / (power-of-two scale of wpk)
    int n, group;         // patches, patches per image
    int prof_id;          // developer role profiler slot
    const int* count;     // valid patches per image (NULL: all)
};

// SA: input hi/lo planes (2: the lo planes arrive as bytes); SW: weight hi/lo copies; OSA: write hi/lo planes (2: lo as bytes).  OUT: layout of the output buffer.  EW: epilogue warps (4 | 8 | 16).
template <int CIN, int COUT, int H, int STRIDE, int NSPLIT, int STAGES, int OUT, int SA, int SW, int OSA, int EW>
struct XCfg {
    using In = XIn<H, STRIDE>;
    static constexpr int KC = CIN / 8, NT = COUT / NSPLIT, HOUT = In::HOUT;
    static constexpr int HAS_LO = SA ? 1 : 0, LO8 = (SA == 2) ? 1 : 0;      // SA = 2: the residual planes arrive as bytes
    static constexpr int G = KC * (1 + HAS_LO);                               // channel groups of one unit (in shared memory)
    static constexpr int GS = STAGES * In::SLOT_STAGE + (STRIDE == 1 ? In::RW : 0);   // slots per channel group in shared memory
    static constexpr int ACCW = 3 * NT;                                        // accumulator columns of one tile
    static constexpr int NACC = (512 / ACCW) < 4 ? (512 / ACCW) : 4;
    static constexpr uint32_t W_BYTES = 9u * CIN * NT * 2u * (1 + SW);         // per split
    static constexpr uint32_t IN_BYTES = (uint32_t)G * GS * 16u;               // all stages
    static constexpr uint32_t HI_IN_BYTES = (uint32_t)KC * In::NPLANES * In::DATA * 16u;
    static constexpr uint32_t UNIT_IN_BYTES = HI_IN_BYTES + (SA == 1 ? HI_IN_BYTES : SA == 2 ? HI_IN_BYTES / 2 : 0u);   // one unit in HBM
    static constexpr int NCONV = 4;                                            // LO8: converter warps (one alone was the new critical path: 32 dependent steps per unit)
    static constexpr int THREADS = 64 + 32 * EW + 32 * NCONV * LO8;
    static constexpr size_t SMEM = 1024 + (size_t)W_BYTES + IN_BYTES;
    static constexpr size_t HI_OUT_BYTES = (size_t)(COUT / 8) * layout_slots(OUT) * 16;
    static constexpr size_t UNIT_OUT_BYTES = (OUT == L_HEAD) ? 0 : HI_OUT_BYTES + (OSA == 1 ? HI_OUT_BYTES : OSA == 2 ? HI_OUT_BYTES / 2 : 0);
    // weight rows per K group of one (dy, k step) block
    static constexpr int NR1 = (1 + SW) * 3 * NT;                              // stride 1: [hi: dx0 dx1 dx2][lo: dx0 dx1 dx2]
    static constexpr int NRO = (1 + SW) * 2 * NT, NRE = (1 + SW) * NT;         // stride 2: odd-x plane [hi: dx0 dx2][lo: ...], even-x plane [hi: dx1][lo: dx1]
    static_assert(CIN % 16 == 0 && NT % 16 == 0 && ACCW <= 256 && NACC >= 2, "UMMA shape");
    static_assert(EW == 4 || EW == 8 || EW == 16, "epilogue warps");
    static constexpr int CS = (EW == 16) ? 2 : 1;     // EW = 16: two tile sets x two column halves (an accumulator is read by 8 warps)
    static_assert((NT / 16) % CS == 0, "column split");
    static_assert(3 * STAGES + 2 * NACC + 1 <= 60, "barrier area");
    static_assert(!LO8 || (STRIDE == 2 && In::DATA % 64 == 0), "byte residual planes: stride-2 consumers");
    static_assert(OSA != 2 || OUT == L_S2_16 || OUT == L_S2_8P, "byte residual planes are written for stride-2 consumers");
    static_assert(SMEM <= 232448, "shared memory budget");
    static_assert(GS < 16384, "leading-byte offset field");
    static_assert(OUT == L_HEAD || layout_pair(OUT) || !In::PAIR, "a pair layer writes pair layouts or the head operand");
};

// MC = 1 (NSPLIT = 2 only): the two CTAs of a unit form a thread-block cluster (1 x 2); each loader fetches half of the unit's planes and
// multicasts them to both, so the input crosses the L2 -> SM fabric once instead of twice (HardNet layer 5 waited for its input 40 % of the time).
template <int CIN, int COUT, int H, int STRIDE, int NSPLIT, int STAGES, int OUT, int SA, int SW, int OSA, int EW, int BF = 0, int MC = 0>
__global__ void __launch_bounds__(64 + 32 * EW + (SA == 2 ? 128 : 0), 1) tcx_conv_kernel(const XArgs a) {
    static_assert(MC == 0 || NSPLIT == 2, "multicast pairs the two channel-split CTAs");
    using Cfg = XCfg<CIN, COUT, H, STRIDE, NSPLIT, STAGES, OUT, SA, SW, OSA, EW>;
    using In = typename Cfg::In;
    constexpr int KC = Cfg::KC, NT = Cfg::NT, NACC = Cfg::NACC, TILES = In::TILES, HOUT = Cfg::HOUT, GS = Cfg::GS, RW = In::RW, W = In::W;
    constexpr int PAIR = In::PAIR;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);  // [STAGES]
    uint64_t* empty = full + STAGES;                       // [STAGES]
    uint64_t* tfull = empty + STAGES;                      // [NACC]
    uint64_t* tempty = tfull + NACC;                       // [NACC]
    uint64_t* wbar = tempty + NACC;
    uint64_t* cfull = wbar + 1;                            // [STAGES] byte planes of the stage expanded (LO8)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(cfull + STAGES);
    constexpr int LO8 = Cfg::LO8;
    static_assert(!(BF && (SA == 2 || OSA == 2)), "byte residual planes are fp16");
    float* s_bias = reinterpret_cast<float*>(smem + 512);  // [NT]
    unsigned char* sW = smem + 1024;
    unsigned char* sIn = sW + Cfg::W_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int split = blockIdx.y;
    const int n_units = PAIR ? (a.n + 1) >> 1 : a.n;

    if (threadIdx.x < NT) s_bias[threadIdx.x] = a.bias[split * NT + threadIdx.x];
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1 + MC); mbar_init(&cfull[s], Cfg::NCONV); }   // MC: both CTAs' MMAs must have read a stage
        for (int i = 0; i < NACC; i++) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4 * Cfg::CS); }
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // zero rows of every stage: written once, the loader only ever writes data rows
    for (int i = threadIdx.x; i < (int)(Cfg::IN_BYTES / 16); i += blockDim.x) reinterpret_cast<uint4*>(sIn)[i] = make_uint4(0, 0, 0, 0);
    if (warp == EW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (MC) cluster_sync();      // the peer's barriers are initialised before anything is multicast into this CTA
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    auto pvalid = [&](int pi) -> bool { return pi < a.n && (a.count == nullptr || (pi % a.group) < a.count[pi / a.group]); };
    auto uvalid = [&](int u) -> bool { return PAIR ? (pvalid(2 * u) || pvalid(2 * u + 1)) : pvalid(u); };

    if (warp == EW) {
        // ===== loader =====
        if (lane == 0) {
            mbar_expect_tx(wbar, Cfg::W_BYTES);
            bulk_g2s(sW, reinterpret_cast<const unsigned char*>(a.wpk) + (size_t)split * Cfg::W_BYTES, Cfg::W_BYTES, wbar);
            int it = 0;
            RP_DECL;
            for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
                if (!uvalid(u)) continue;
                const int s = it % STAGES;
                RP_WAIT(0, mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1));
                mbar_expect_tx(&full[s], Cfg::UNIT_IN_BYTES);
                const unsigned char* gsrc = reinterpret_cast<const unsigned char*>(a.in) + (size_t)u * Cfg::UNIT_IN_BYTES;
#pragma unroll 1
                for (int g = 0; g < Cfg::G; g++)
#pragma unroll
                    for (int pl = 0; pl < In::NPLANES; pl++) {
                        unsigned char* dst = sIn + ((size_t)g * GS + (size_t)s * In::SLOT_STAGE + (size_t)pl * In::PLANE + RW) * 16;
                        const unsigned char* srcp = gsrc + ((size_t)g * In::NPLANES + pl) * In::DATA * 16;
                        if (LO8 && g >= KC) {   // byte plane: into the upper half of the fp16 plane's place, expanded there by the converter warp
                            bulk_g2s(dst + In::DATA * 8, gsrc + Cfg::HI_IN_BYTES + ((size_t)(g - KC) * In::NPLANES + pl) * In::DATA * 8, In::DATA * 8u, &full[s]);
                        } else if (MC) { if (((g * In::NPLANES + pl) & 1) == split) bulk_g2s_mc(dst, srcp, In::DATA * 16u, &full[s], (uint16_t)3); }
                        else bulk_g2s(dst, srcp, In::DATA * 16u, &full[s]);
                    }
                it++;
            }
            if (MC) {   // drain: the peer's last commits on this CTA's `empty` barriers must have landed before the CTA may exit
                for (int k = 0; k < STAGES && k < it; k++) { const int j = it - 1 - k; mbar_wait(&empty[j % STAGES], (j / STAGES) & 1); }
            }
            XP_STORE(a.prof_id, 3);
        }
    } else if (warp == EW + 1) {
        // ===== MMA issuer (warp-uniform control flow, one elected lane issues) =====
        constexpr uint32_t idesc3 = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)((3 * NT) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t leader = elect_one();
        mbar_wait(wbar, 0);
        tc_fence_after();
        const uint32_t w_base = smem_u32(sW) >> 4;           // 16-byte units
        const uint32_t in_base = smem_u32(sIn) >> 4;
        constexpr uint32_t LBO_A = ((uint32_t)GS) << 16;      // (bytes >> 4) << 16
        int it = 0, tcnt = 0;
        RP_DECL;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
            if (!uvalid(u)) continue;
            const int s = it % STAGES;
            RP_WAIT(0, mbar_wait(LO8 ? &cfull[s] : &full[s], (it / STAGES) & 1));
            tc_fence_after();
            const uint32_t st_base = in_base + (uint32_t)(s * In::SLOT_STAGE);
#pragma unroll 1
            for (int t = 0; t < TILES; t++, tcnt++) {
                const int ab = tcnt % NACC;
                RP_WAIT(1, mbar_wait(&tempty[ab], ((tcnt / NACC) & 1) ^ 1));
                tc_fence_after();
                if (leader) {
                    const uint32_t d = tmem + (uint32_t)(ab * Cfg::ACCW);
                    const uint32_t a_t = st_base + (uint32_t)(t * 128);
                    if (STRIDE == 1) {
#pragma unroll
                        for (int dy = 0; dy < 3; dy++) {
#pragma unroll
                            for (int j = 0; j < KC / 2; j++) {
                                const uint32_t ahi = ((a_t + (uint32_t)(dy * RW + 2 * j * GS)) & 0x3FFFu) | LBO_A;
                                const uint32_t alo = ((a_t + (uint32_t)(dy * RW + (KC + 2 * j) * GS)) & 0x3FFFu) | LBO_A;
                                const uint32_t blk = w_base + (uint32_t)((dy * (KC / 2) + j) * 2 * Cfg::NR1);
                                const uint32_t bhi = (blk & 0x3FFFu) | ((uint32_t)Cfg::NR1 << 16), blo = ((blk + 3 * NT) & 0x3FFFu) | ((uint32_t)Cfg::NR1 << 16);
                                if (dy == 0 && j == 0) umma_f16_lo<0>(d, ahi, bhi, idesc3); else umma_f16_lo<1>(d, ahi, bhi, idesc3);
                                if (SW) umma_f16_lo<1>(d, ahi, blo, idesc3);
                                if (SA) umma_f16_lo<1>(d, alo, bhi, idesc3);
                            }
                        }
                    } else {
                        xmma_s2_tile<KC, NT, In::PLANE, RW, GS, SA, SW, BF>(d, a_t, w_base);
                    }
                    umma_commit(&tfull[ab]);
                }
                __syncwarp();
            }
            if (leader) { if (MC) umma_commit_mc(&empty[s], (uint16_t)3); else umma_commit(&empty[s]); }
            __syncwarp();
            it++;
        }
        XP_STORE(a.prof_id, 0);
    } else if (LO8 && warp >= EW + 2) {
        // ===== converters (NCONV warps, regions dealt round robin): byte residual planes -> fp16 in place (byte j of a slot pair becomes the
        // fp16 with that high byte).  The bytes sit in the upper half of the plane's place; a warp reads a whole region (16 bytes per lane and
        // step) into registers before it writes the expanded 32 bytes per lane and step, so nothing is overwritten before it is read =====
        constexpr int NST = In::DATA / 64;                    // steps of 32 lanes x 16 bytes per region
        const int cw = warp - (EW + 2);
        int it = 0;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
            if (!uvalid(u)) continue;
            const int s = it % STAGES;
            mbar_wait(&full[s], (it / STAGES) & 1);
#pragma unroll 1
            for (int r = cw; r < KC * In::NPLANES; r += Cfg::NCONV) {
                const int g = KC + r / In::NPLANES, pl = r % In::NPLANES;
                unsigned char* region = sIn + ((size_t)g * GS + (size_t)s * In::SLOT_STAGE + (size_t)pl * In::PLANE + RW) * 16;
                uint4 b[NST];
#pragma unroll
                for (int k = 0; k < NST; k++) b[k] = *reinterpret_cast<const uint4*>(region + In::DATA * 8 + (k * 32 + lane) * 16);
                __syncwarp();
#pragma unroll
                for (int k = 0; k < NST; k++) {
                    *reinterpret_cast<uint4*>(region + (k * 32 + lane) * 32) =
                        make_uint4(__byte_perm(b[k].x, 0u, 0x1404), __byte_perm(b[k].x, 0u, 0x3424), __byte_perm(b[k].y, 0u, 0x1404), __byte_perm(b[k].y, 0u, 0x3424));
                    *reinterpret_cast<uint4*>(region + (k * 32 + lane) * 32 + 16) =
                        make_uint4(__byte_perm(b[k].z, 0u, 0x1404), __byte_perm(b[k].z, 0u, 0x3424), __byte_perm(b[k].w, 0u, 0x1404), __byte_perm(b[k].w, 0u, 0x3424));
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&cfull[s]);
            it++;
        }
    } else {
        // ===== epilogue: EW / 4 sets of four warps (TMEM lane quadrant = warp % 4), set k takes tiles k, k + NSETS, ... =====
        constexpr int CS = Cfg::CS, NSETS = EW / 4 / CS;    // tile sets; each made of CS column parts of four warps
        const int q = warp & 3;
        const int set = (warp >> 2) / CS, cpart = (warp >> 2) % CS;
        const int r = q * 32 + lane;                         // tile row of this thread
        int tcnt = 0;
        RP_DECL;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
            if (!uvalid(u)) continue;
#pragma unroll 1
            for (int t = 0; t < TILES; t++, tcnt++) {
                if ((tcnt % NSETS) != set) continue;
                const int ab = tcnt % NACC;
                RP_WAIT(0, mbar_wait(&tfull[ab], (tcnt / NACC) & 1));
                tc_fence_after();
                // pixel of this row
                int y, x, p, pi;
                if (PAIR) { y = r >> 4; p = (r >> 3) & 1; x = r & 7; pi = 2 * u + p; }
                else { const int m = t * 128 + r; y = m / W; x = m - y * W; p = u & 1; pi = u; }
                const bool ok = pvalid(pi);
                const float mask_l = x > 0 ? 1.f : 0.f, mask_r = x < W - 1 ? 1.f : 0.f;
                const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACCW);
                // output position
                unsigned char* obase = nullptr;
                unsigned char* obase8 = nullptr;     // OSA = 2: byte residual planes behind the hi planes
                size_t lo_off = 0;
                if (OUT == L_HEAD) {
                    obase = reinterpret_cast<unsigned char*>(a.out) + (((size_t)(pi >> 7) * (HOUT * HOUT * COUT / 8) + (size_t)(y * HOUT + x) * (COUT / 8)) * 128 + (pi & 127)) * 16;
                    lo_off = (size_t)((a.n + 127) >> 7) * (HOUT * HOUT * COUT / 8) * 128 * 16;
                } else {
                    const int ou = layout_pair(OUT) ? (pi >> 1) : pi;
                    obase = reinterpret_cast<unsigned char*>(a.out) + (size_t)ou * Cfg::UNIT_OUT_BYTES + (size_t)layout_slot(OUT, y, x, pi & 1) * 16;
                    lo_off = (size_t)(COUT / 8) * layout_slots(OUT) * 16;
                    obase8 = reinterpret_cast<unsigned char*>(a.out) + (size_t)ou * Cfg::UNIT_OUT_BYTES + Cfg::HI_OUT_BYTES + (size_t)layout_slot(OUT, y, x, pi & 1) * 8;
                }
#pragma unroll 1
                for (int c0 = cpart * 16; c0 < NT; c0 += 16 * CS) {
                    uint32_t r0[16], r1[16], r2[16];
                    tmem_ld16(taddr + (uint32_t)c0, r0);                   // stride 1: dx0 | stride 2: odd plane dx0
                    tmem_ld16(taddr + (uint32_t)(NT + c0), r1);            // stride 1: dx1 | stride 2: odd plane dx2
                    tmem_ld16(taddr + (uint32_t)(2 * NT + c0), r2);        // stride 1: dx2 | stride 2: even plane dx1
                    tmem_ld_wait();
                    if (c0 + 16 * CS >= NT) {   // this warp's last column chunk read: release the accumulator buffer (4 CS arrivals)
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty[ab]);
                    }
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        // the neighbour outside the image row is the zero padding: multiply by a 0/1 mask (one FFMA instead of select + add)
                        const float left = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[i]), 1, W);
                        float acc;
                        if (STRIDE == 1) {
                            const float right = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[i]), 1, W);
                            acc = fmaf(left, mask_l, fmaf(right, mask_r, __uint_as_float(r1[i])));
                        } else {
                            acc = fmaf(left, mask_l, __uint_as_float(r1[i]) + __uint_as_float(r2[i]));
                        }
                        v[i] = fmaxf(fmaf(acc, a.inv_scale, s_bias[c0 + i]), 0.f);
                    }
                    if (ok) {
#pragma unroll
                        for (int g = 0; g < 2; g++) {
                            const int cg = (split * NT + c0) / 8 + g;       // channel group of the output
                            const size_t goff = (OUT == L_HEAD) ? (size_t)cg * 128 * 16 : (size_t)cg * layout_slots(OUT) * 16;
                            uint4 hi, lo;
                            split_pack8<OSA, BF>(v + g * 8, hi, lo);
                            *reinterpret_cast<uint4*>(obase + goff) = hi;
                            if (OSA == 1) *reinterpret_cast<uint4*>(obase + lo_off + goff) = lo;
                            if (OSA == 2) *reinterpret_cast<uint2*>(obase8 + (size_t)cg * layout_slots(OUT) * 8) = pack_lo8(lo);
                        }
                    }
                }
            }
        }
        if (warp == 0) XP_STORE(a.prof_id, 1);
    }
    tc_fence_before();
    __syncthreads();
    if (MC) cluster_sync();      // neither CTA leaves while the other may still signal its barriers
    if (warp == EW + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
    }
}

}  // namespace tcx
}  // namespace ag
