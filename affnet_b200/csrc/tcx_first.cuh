// First two conv layers of AffNet / OriNet / HardNet in ONE kernel, second-generation formulation (see tcx_conv.cuh):
//
//   sampler (LAF.py:313-372) -> input_norm (architectures.py:231-235) -> conv3x3(1 -> C1)+BN+ReLU -> conv3x3(C1 -> COUT)+BN+ReLU
//
// 32x32 patches and the layer-1 activations never exist in HBM.  Tiles are 128 consecutive pixels = 4 image rows of 32 (8 tiles per
// patch, no padded columns).  Layer 1 (K = 9): the sliding-window plane P[y*32 + x] = {4 pixels of padded row y from column x | 4
// pixels of padded row y+1} makes one M=128, K=16 MMA cover kernel rows 0 and 1, the same plane two rows further (descriptor
// leading-byte offset) kernel row 2.  Layer 2: for kernel row dy one MMA over the layer-1 stage advanced by dy rows with the three
// taps of that row stacked along N (N = 3*COUT, or 6*COUT with the weight residual stacked behind when that still fits N = 96);
// the epilogue shifts the dx = 0 / dx = 2 blocks by one pixel with warp shuffles (a warp = one image row).
// Split precision: the input and layer-1 weights always carry fp16 residual planes; SA / SW / OSA as in tcx_conv.cuh.
//
// Warp roles (21 warps; 25 for 32-channel nets), ordered by the scheduler's priority (the SMSP arbiter prefers the highest warp id,
// B300_MICROARCH.md): last warp MMA issuer (+ TMEM, weights) | the four below it layer-1 epilogue (TMEM -> bias/ReLU -> fp16 stage in
// shared memory) | from warp 8 the layer-2 epilogue, NSET sets of four taking tiles in turn (TMEM -> shuffles -> bias/ReLU -> fp16 ->
// global, stride-2 consumer layout) | 0-7 sampler + input_norm + P planes.
//
// L3 = 1 (AffNet / OriNet): conv layer 3 (16 -> 32, stride 2) runs in the same kernel.  Layer 2's output (16 x 32x32, fp16 hi + lo,
// 64 KiB per patch, the largest activation of the net) then never crosses HBM: the layer-2 epilogue writes it into shared memory as
// the four parity planes tcx_conv's loader builds for a stride-2 consumer (XIn<32, 2>), the issuer adds layer 3's two tiles with the
// same MMA sequence as tcx_conv (xmma_s2_tile), and four more epilogue warps (8-11, below the layer-2 sets) apply tcx_conv's stride-2
// epilogue arithmetic and write the L_S1_16 planes layer 4 reads.  Same MMAs, same order, same epilogue: bit-identical to the pair
// tcx_first_kernel + tcx_conv_kernel.  Shared memory: the layer-3 input (68 KiB) and weights (18 KiB) fit because both the layer-2
// stage and the layer-3 input are single-buffered with barriers per tile (a stage tile is refilled as soon as the MMAs that read it are
// done) instead of double-buffered per patch.
#pragma once
#include "tcx_conv.cuh"

namespace ag {
namespace tcx {

template <int C1, int COUT, int SA, int SW, int OSA, int L3 = 0>
struct XFirstCfg {
    static constexpr int KC = C1 / 8, NT = COUT;
    static constexpr int TILES = 8;
    static constexpr int NPIXP = 18 * 32;                      // slots of one HALF P plane: 18 window rows (16 image rows of outputs + 2 rows of look-ahead)
    static constexpr int SX = 1200;                            // floats of one padded fp32 patch buffer: 34*34 + zero tail (windows of row 33 look one row further)
    static constexpr int S1 = (C1 == 16) ? 1 : 0;              // layer 1: x_hi * [w_hi ; w_lo] as one N = 2*C1 MMA
    static constexpr int ACC1 = 32;                            // layer-1 accumulator columns per tile (2*16 stacked, or 32)
    static constexpr int NL1 = 4;                              // layer-1 accumulator buffers
#ifndef AG_FIRST_STACK
#define AG_FIRST_STACK 0   // measured (r02): stacking [W_hi ; W_lo] along N saves a third of the MMAs but its extra TMEM reads and hi + lo adds make the layer-2 epilogue the
                           // critical role: 7.2k -> 7.5k clk per patch (AffNet / OriNet), 10.3k -> 12.8k (HardNet, only two accumulator buffers left)
#endif
    static constexpr int STACK = (AG_FIRST_STACK && SW && 6 * NT <= 192) ? 1 : 0; // layer 2: [W_hi ; W_lo] stacked along N
    static constexpr int ACCW = 3 * NT * (1 + STACK);
    // fused layer 3: 16 -> 2 COUT channels, stride 2, two tiles of 8 output rows; one accumulator buffer per tile
    using In3 = XIn<32, 2>;
    static constexpr int NT3 = L3 ? 2 * COUT : 0, KC3 = COUT / 8, G3 = 2 * KC3, GS3 = In3::SLOT_STAGE;
    static constexpr int ACCW3 = 3 * NT3;
    static constexpr int ACC3_COLS = L3 ? In3::TILES * ACCW3 : 0;
    static constexpr int NACC = (512 - NL1 * ACC1 - ACC3_COLS) / ACCW < 4 ? (512 - NL1 * ACC1 - ACC3_COLS) / ACCW : 4;
    static constexpr int G = KC * (1 + SA);
    static constexpr int SLOT_STAGE = 1024 + 32;               // zero row + 32 data rows; the zero row below is the next stage's / the trailing one
    static constexpr int STAGES = L3 ? 1 : 2;                  // layer-2 stages (L3: one, refilled tile by tile)
    static constexpr int GS = STAGES * SLOT_STAGE + 32;
    static constexpr int NR = (1 + SW) * 3 * NT;               // weight rows per K group of a (dy, k step) block
    static constexpr uint32_t W_BYTES = 9u * C1 * NT * 2u * (1 + SW);
    static constexpr uint32_t IN_BYTES = (uint32_t)G * GS * 16u;
    static constexpr uint32_t W1_BYTES = 2u * 2u * C1 * 16;    // [K chunk 0|1][hi rows | lo rows][8]
    static constexpr uint32_t P_BYTES = 2u * 2u * NPIXP * 16;   // [half][hi | lo][NPIXP]: the halves are built and consumed alternately
    static constexpr uint32_t W3_BYTES = L3 ? 9u * COUT * NT3 * 2u * 2u : 0u;      // layer-3 weights, hi + lo copies
    static constexpr uint32_t IN3_BYTES = L3 ? (uint32_t)G3 * GS3 * 16u : 0u;      // layer-3 input: [hi | lo groups][4 parity planes][zero row | 256]
    static constexpr size_t UNIT_OUT3_BYTES = (size_t)2 * (NT3 / 8) * 256 * 16;   // layer-3 output (L_S1_16, hi + lo)
    static constexpr size_t SMEM = 1024 + (size_t)W_BYTES + IN_BYTES + P_BYTES + W1_BYTES + 2 * SX * 4 + 256 + W3_BYTES + IN3_BYTES;
    static constexpr size_t HI_OUT_BYTES = (size_t)(COUT / 8) * 1024 * 16;
    static constexpr size_t UNIT_OUT_BYTES = HI_OUT_BYTES + (OSA == 1 ? HI_OUT_BYTES : OSA == 2 ? HI_OUT_BYTES / 2 : 0);   // OSA = 2: byte residual planes
#ifndef AG_FIRST_NSET16
#define AG_FIRST_NSET16 2   // three sets measured slower for the 16-channel nets (4.05 -> 4.28 ms per step over the three first kernels)
#endif
    static constexpr int NSET = (C1 >= 32) ? 3 : AG_FIRST_NSET16;            // layer-2 epilogue sets of four warps (HardNet's 32-channel epilogue is its critical role: three sets)
    static constexpr int W_L3 = 8, W_L2 = W_L3 + 4 * L3, W_L1 = W_L2 + 4 * NSET, W_MMA = W_L1 + 4;   // first warp of each role (producers: warps 0-7)
    static constexpr int THREADS = (W_MMA + 1) * 32;
    static_assert(C1 % 16 == 0 && NT % 16 == 0 && NACC >= 2 && ACCW <= 256, "shape");
    static_assert(C1 == 16 || C1 == 32, "layer-1 accumulator width");
    static_assert(SMEM <= 232448, "shared memory budget");
    static_assert(!L3 || (C1 == 16 && COUT == 16 && SA == 1 && SW == 1 && OSA == 1), "fused layer 3: the 16-channel nets with fp16 residual planes");
    static_assert(!L3 || (In3::TILES == 2 && GS3 < 16384), "layer-3 tiles");
};

// a3 (L3 = 1): layer 3's weights, bias, scale and output buffer; a.out is then unused
template <int C1, int COUT, int SA, int SW, int OSA, int BF = 0, int L3 = 0>
__global__ void __launch_bounds__(XFirstCfg<C1, COUT, SA, SW, OSA, L3>::THREADS, 1) tcx_first_kernel(const XArgs a, const FirstSrc src, const XArgs a3) {
    using Cfg = XFirstCfg<C1, COUT, SA, SW, OSA, L3>;
    using In3 = typename Cfg::In3;
    constexpr int KC = Cfg::KC, NT = Cfg::NT, NACC = Cfg::NACC, TILES = Cfg::TILES, NPIXP = Cfg::NPIXP, SX = Cfg::SX, GS = Cfg::GS, NL1 = Cfg::NL1;
    constexpr int NT3 = Cfg::NT3, GS3 = Cfg::GS3;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);   // [8]   layer-2 stage s filled (128 layer-1 epilogue threads); L3: stage tile t written
    uint64_t* empty = full + 8;                             // [8]   layer-2 MMAs done with stage s; L3: with stage tile t
    uint64_t* tfull = empty + 8;                            // [4]
    uint64_t* tempty = tfull + 4;                           // [4]
    uint64_t* wbar = tempty + 4;
    uint64_t* p_full = wbar + 1;                            // [2] half P plane written (256 producer threads)
    uint64_t* p_empty = p_full + 2;                         // [2] layer-1 MMAs done with the half
    uint64_t* c1_full = p_empty + 2;                        // [4]
    uint64_t* c1_empty = c1_full + 4;                       // [4]
    uint64_t* f3_full = c1_empty + 4;                       // [2]   L3: layer-3 input rows of tile u written (layer-2 epilogue threads)
    uint64_t* f3_empty = f3_full + 2;                       // [2]   L3: layer-3 MMAs of tile u done with their input
    uint64_t* t3_full = f3_empty + 2;                       // [2]   L3: layer-3 accumulator u
    uint64_t* t3_empty = t3_full + 2;                       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t3_empty + 2);   // byte 360
    float* s_bias1 = reinterpret_cast<float*>(smem + 384);  // [C1]
    float* s_bias = reinterpret_cast<float*>(smem + 512);   // [NT]
    float* s_bias3 = reinterpret_cast<float*>(smem + 640);  // [NT3]
    unsigned char* sW = smem + 1024;
    unsigned char* sIn = sW + Cfg::W_BYTES;                 // [G][2 stages][zero row | 32 data rows] + trailing zero row
    unsigned char* sP = sIn + Cfg::IN_BYTES;                // [half][hi|lo][NPIXP][8] fp16
    unsigned char* sW1 = sP + Cfg::P_BYTES;                 // [chunk][hi|lo][C1][8] fp16
    float* s_x = reinterpret_cast<float*>(sW1 + Cfg::W1_BYTES);   // [2][SX]
    float* s_red = s_x + 2 * SX;                            // [2][8][2]
    unsigned char* sW3 = reinterpret_cast<unsigned char*>(s_x + 2 * SX) + 256;   // L3: layer-3 weights (tcx_pack_layer, stride 2)
    unsigned char* sIn3 = sW3 + Cfg::W3_BYTES;              // L3: [G3][4 parity planes][zero row | 256 data slots]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto valid = [&](int pi) -> bool { return a.count == nullptr || (pi % a.group) < a.count[pi / a.group]; };
    auto next_valid = [&](int pi) -> int {
        while (pi < a.n && !valid(pi)) pi += gridDim.x;
        return pi;
    };

    // ---- one-time setup by all threads ----
    if (threadIdx.x < NT) s_bias[threadIdx.x] = a.bias[threadIdx.x];
    if (threadIdx.x < C1) s_bias1[threadIdx.x] = src.b1[threadIdx.x];
    if (L3 && threadIdx.x < NT3) s_bias3[threadIdx.x] = a3.bias[threadIdx.x];
    if (threadIdx.x == 0) {
        for (int s = 0; s < (L3 ? TILES : 2); s++) { mbar_init(&full[s], 128); mbar_init(&empty[s], 1); }
        for (int i = 0; i < 4; i++) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); mbar_init(&c1_full[i], 1); mbar_init(&c1_empty[i], 4); }
        if (L3) {   // layer-3 tile 0 reads layer-2 rows 0..15 (layer-2 tiles 0-3), tile 1 rows 15..31 (tiles 3-7): 128 arrivals per layer-2 tile
            mbar_init(&f3_full[0], 4 * 128); mbar_init(&f3_full[1], 5 * 128);
            for (int u = 0; u < 2; u++) { mbar_init(&f3_empty[u], 1); mbar_init(&t3_full[u], 1); mbar_init(&t3_empty[u], 4); }
        }
        mbar_init(wbar, 1);
        for (int hh = 0; hh < 2; hh++) { mbar_init(&p_full[hh], 256); mbar_init(&p_empty[hh], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < 2 * 2 * C1 * 8; i += blockDim.x) {   // W1[chunk][hi rows | lo rows][e]: chunk 0 = kernel rows 0 (e 0..2), 1 (e 4..6); chunk 1 = kernel row 2
        const int e = i & 7, co = (i >> 3) % C1, part = (i / (8 * C1)) & 1, ch = i / (8 * C1 * 2);
        const int dy = ch == 0 ? (e >> 2) : 2, dx = e & 3;
        float v = 0.f;
        if (dx < 3 && (ch == 0 || e < 4)) {
            const float wv = src.w1[(dy * 3 + dx) * C1 + co] * src.w1_scale;   // power-of-two scale, undone in the epilogue
            const float hi = unpack2<BF>(pack2<BF>(wv, 0.f)).x;      // wv rounded to the operand format
            v = part == 0 ? hi : wv - hi;
        }
        reinterpret_cast<unsigned short*>(sW1)[i] = (unsigned short)(pack2<BF>(v, 0.f) & 0xFFFFu);
    }
    for (int i = threadIdx.x; i < (int)((Cfg::IN_BYTES + Cfg::P_BYTES) / 16); i += blockDim.x) reinterpret_cast<uint4*>(sIn)[i] = make_uint4(0, 0, 0, 0);
    for (int i = threadIdx.x; i < 2 * SX; i += blockDim.x) s_x[i] = 0.f;
    for (int i = threadIdx.x; i < (int)(Cfg::IN3_BYTES / 16); i += blockDim.x) reinterpret_cast<uint4*>(sIn3)[i] = make_uint4(0, 0, 0, 0);   // zero rows
    if (warp == Cfg::W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tmem_l2 = tmem + (uint32_t)(NL1 * Cfg::ACC1);
    const uint32_t tmem_l3 = tmem_l2 + (uint32_t)(NACC * Cfg::ACCW);

    if (warp == Cfg::W_MMA) {
        // ===== MMA issuer: layer 1 runs one patch ahead of layer 2 =====
        constexpr uint32_t idesc_all = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)(Cfg::ACCW >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);      // N = 3 NT (or 6 NT stacked)
        constexpr uint32_t idesc_3 = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)((3 * NT) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        constexpr uint32_t idesc1 = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)(C1 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        constexpr uint32_t idesc1_st = XFmt<BF>::IDESC | (1u << 4) | ((uint32_t)((2 * C1) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t leader = elect_one();
        if (leader) {
            mbar_expect_tx(wbar, Cfg::W_BYTES + Cfg::W3_BYTES);
            bulk_g2s(sW, a.wpk, Cfg::W_BYTES, wbar);
            if (L3) bulk_g2s(sW3, a3.wpk, Cfg::W3_BYTES, wbar);
        }
        __syncwarp();
        mbar_wait(wbar, 0);
        tc_fence_after();
        const uint32_t w_base = smem_u32(sW) >> 4, in_base = smem_u32(sIn) >> 4, w3_base = smem_u32(sW3) >> 4, in3_base = smem_u32(sIn3) >> 4;
        const uint32_t w1_lo = desc_lo(smem_u32(sW1), 2 * C1 * 16u);       // K chunks are 2*C1 rows apart (hi rows, then lo rows)
        const uint32_t p_lo = desc_lo(smem_u32(sP), 2 * 32 * 16u);          // leading-byte offset = two image rows
        constexpr uint32_t LBO_A = ((uint32_t)GS) << 16;
        int c1cnt = 0, tcnt = 0;
        RP_DECL;
        auto l1_tile = [&](int t) {
            const int b = c1cnt % NL1;
            RP_WAIT(1, mbar_wait(&c1_empty[b], ((c1cnt / NL1) & 1) ^ 1));
            tc_fence_after();
            if (leader) {
                const uint32_t d = tmem + (uint32_t)(b * Cfg::ACC1);
                const uint32_t alo = p_lo + (uint32_t)((t >> 2) * 2 * NPIXP + (t & 3) * 128);   // half t/4, tile t%4 of it
                if (Cfg::S1) {   // x_hi * [w_hi ; w_lo] in one MMA, then x_lo * w_hi
                    umma_f16_lo<0>(d, alo, w1_lo, idesc1_st);
                    umma_f16_lo<1>(d, alo + (uint32_t)NPIXP, w1_lo, idesc1);
                } else {
                    umma_f16_lo<0>(d, alo, w1_lo, idesc1);
                    umma_f16_lo<1>(d, alo + (uint32_t)NPIXP, w1_lo, idesc1);             // x_lo * w_hi
                    umma_f16_lo<1>(d, alo, w1_lo + (uint32_t)C1, idesc1);                 // x_hi * w_lo (lo rows follow the hi rows)
                }
                umma_commit(&c1_full[b]);
            }
            __syncwarp();
            c1cnt++;
        };
        auto l2_tile = [&](uint32_t st_base, int t) {
            const int ab = tcnt % NACC;
            RP_WAIT(3, mbar_wait(&tempty[ab], ((tcnt / NACC) & 1) ^ 1));
            tc_fence_after();
            if (leader) {
                const uint32_t d = tmem_l2 + (uint32_t)(ab * Cfg::ACCW);
                const uint32_t a_t = st_base + (uint32_t)(t * 128);
#pragma unroll
                for (int dy = 0; dy < 3; dy++) {
#pragma unroll
                    for (int j = 0; j < KC / 2; j++) {
                        const uint32_t ahi = ((a_t + (uint32_t)(dy * 32 + 2 * j * GS)) & 0x3FFFu) | LBO_A;
                        const uint32_t alo = ((a_t + (uint32_t)(dy * 32 + (KC + 2 * j) * GS)) & 0x3FFFu) | LBO_A;
                        const uint32_t blk = w_base + (uint32_t)((dy * (KC / 2) + j) * 2 * Cfg::NR);
                        const uint32_t bhi = (blk & 0x3FFFu) | ((uint32_t)Cfg::NR << 16), blo = ((blk + 3 * NT) & 0x3FFFu) | ((uint32_t)Cfg::NR << 16);
                        if (Cfg::STACK) {   // A_hi * [W_hi ; W_lo] (N = 6 NT), then A_lo * W_hi into the hi columns
                            if (dy == 0 && j == 0) umma_f16_lo<0>(d, ahi, bhi, idesc_all); else umma_f16_lo<1>(d, ahi, bhi, idesc_all);
                            if (SA) umma_f16_lo<1>(d, alo, bhi, idesc_3);
                        } else {
                            if (dy == 0 && j == 0) umma_f16_lo<0>(d, ahi, bhi, idesc_3); else umma_f16_lo<1>(d, ahi, bhi, idesc_3);
                            if (SW) umma_f16_lo<1>(d, ahi, blo, idesc_3);
                            if (SA) umma_f16_lo<1>(d, alo, bhi, idesc_3);
                        }
                    }
                }
                umma_commit(&tfull[ab]);
            }
            __syncwarp();
            tcnt++;
        };
        // L3: layer-3 tile u of the k-th patch (its input rows written by the layer-2 epilogue, its accumulator drained)
        auto l3_tile = [&](int u, int k) {
            RP_WAIT(2, mbar_wait(&f3_full[u], k & 1));
            RP_WAIT(3, mbar_wait(&t3_empty[u], (k & 1) ^ 1));
            tc_fence_after();
            if (leader) {
                xmma_s2_tile<Cfg::KC3, NT3, In3::PLANE, In3::RW, GS3, 1, 1, BF>(tmem_l3 + (uint32_t)(u * Cfg::ACCW3), in3_base + (uint32_t)(u * 128), w3_base);
                umma_commit(&t3_full[u]);
                umma_commit(&f3_empty[u]);
            }
            __syncwarp();
        };
        // layer 1 of patch i+1 is issued tile by tile between the layer-2 tiles of patch i: both epilogues are fed at a steady rate and
        // four layer-1 accumulator buffers are enough
        // The P plane lives in two halves (tiles 0-3 / 4-7) with their own barriers: while the layer-1 MMAs of one half run the producers
        // build the other, so the issuer never waits for a whole plane.
        // (two nested loops over half and tile-in-half: indexing the barriers with t >> 2 under (t & 3) guards was miscompiled by nvcc 12.9 -
        // the strength-reduced address of &p_empty[t >> 2] came out as base + 2 t)
        int pi = next_valid(blockIdx.x);
        if (pi < a.n) {
#pragma unroll 1
            for (int hh = 0; hh < 2; hh++) {
                mbar_wait(&p_full[hh], 0);
                tc_fence_after();
#pragma unroll 1
                for (int j = 0; j < 4; j++) l1_tile(hh * 4 + j);
                if (leader) umma_commit(&p_empty[hh]);
                __syncwarp();
            }
        }
        int it = 0;
        while (pi < a.n) {
            const int pn = next_valid(pi + gridDim.x);
            const bool has_next = pn < a.n;
            const int s = L3 ? 0 : (it & 1);
            if (!L3) {
                RP_WAIT(2, mbar_wait(&full[s], (it >> 1) & 1));
                tc_fence_after();
            }
            const uint32_t st_base = in_base + (uint32_t)(s * Cfg::SLOT_STAGE);
#pragma unroll 1
            for (int hh = 0; hh < 2; hh++) {
                if (has_next) { RP_WAIT(0, mbar_wait(&p_full[hh], (it + 1) & 1)); tc_fence_after(); }
#pragma unroll 1
                for (int j = 0; j < 4; j++) {
                    const int t = hh * 4 + j;
                    if (has_next) l1_tile(t);
                    if (L3) {   // layer-2 tile t reads stage rows 4t-1 .. 4t+4: stage tiles t-1 .. t+1, written in order
                        RP_WAIT(2, mbar_wait(&full[t + 1 < TILES ? t + 1 : t], it & 1));
                        tc_fence_after();
                    }
                    l2_tile(st_base, t);
                    if (L3) {
                        // stage tile t-1 is last read by layer-2 tile t: the layer-1 epilogue may refill it for the next patch
                        if (leader) { if (t > 0) umma_commit(&empty[t - 1]); if (t == TILES - 1) umma_commit(&empty[t]); }
                        __syncwarp();
                        // layer 3 two layer-2 tile pairs behind the epilogue whose rows it needs, so the issuer rarely waits for them:
                        // tile 1 of the previous patch (layer-2 rows 15..31) and tile 0 of this one (rows 0..15)
                        if (t == 2 && it > 0) l3_tile(1, it - 1);
                        if (t == 6) l3_tile(0, it);
                    }
                }
                if (has_next) { if (leader) umma_commit(&p_empty[hh]); __syncwarp(); }
            }
            if (!L3) {
                if (leader) umma_commit(&empty[s]);
                __syncwarp();
            }
            it++;
            pi = pn;
        }
        if (L3 && it > 0) l3_tile(1, it - 1);
        XP_STORE(0, 0);
    } else if (warp >= Cfg::W_L2 && warp < Cfg::W_L1) {
        // ===== layer-2 epilogue: TMEM -> x shifts -> bias + ReLU -> fp16 -> global (parity planes of the stride-2 consumer) =====
        const int q = warp & 3, set = (warp - Cfg::W_L2) >> 2;
        const int r = q * 32 + lane;
        const int x = lane;
        const float mask_l = x > 0 ? 1.f : 0.f, mask_r = x < 31 ? 1.f : 0.f;
        float bias2[NT];
#pragma unroll
        for (int i = 0; i < NT; i++) bias2[i] = s_bias[i];
        int tcnt = 0, k = 0;
        RP_DECL;
        for (int pi = next_valid(blockIdx.x); pi < a.n; pi = next_valid(pi + gridDim.x), k++) {
            unsigned char* outp = L3 ? nullptr : reinterpret_cast<unsigned char*>(a.out) + (size_t)pi * Cfg::UNIT_OUT_BYTES;
#pragma unroll 1
            for (int t = 0; t < TILES; t++, tcnt++) {
                if ((tcnt % Cfg::NSET) != set) continue;
                const int ab = tcnt % NACC;
                RP_WAIT(0, mbar_wait(&tfull[ab], (tcnt / NACC) & 1));
                tc_fence_after();
                const int y = t * 4 + q;
                const uint32_t taddr = tmem_l2 + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACCW);
                unsigned char* obase = L3 ? sIn3 + (size_t)(((y & 1) * 2 + (x & 1)) * In3::PLANE + In3::RW + (y >> 1) * 16 + (x >> 1)) * 16
                                          : outp + (size_t)layout_slot(L_S2_16, y, x, 0) * 16;
                (void)r;
#pragma unroll
                for (int c0 = 0; c0 < NT; c0 += 16) {
                    uint32_t r0[16], r1[16], r2[16];
                    if (Cfg::STACK) {   // hi block + A_hi * W_lo block, one tap at a time (registers)
                        uint32_t l[16];
                        tmem_ld16(taddr + (uint32_t)c0, r0); tmem_ld16(taddr + (uint32_t)(3 * NT + c0), l);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; i++) r0[i] = __float_as_uint(__uint_as_float(r0[i]) + __uint_as_float(l[i]));
                        tmem_ld16(taddr + (uint32_t)(NT + c0), r1); tmem_ld16(taddr + (uint32_t)(4 * NT + c0), l);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; i++) r1[i] = __float_as_uint(__uint_as_float(r1[i]) + __uint_as_float(l[i]));
                        tmem_ld16(taddr + (uint32_t)(2 * NT + c0), r2); tmem_ld16(taddr + (uint32_t)(5 * NT + c0), l);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; i++) r2[i] = __float_as_uint(__uint_as_float(r2[i]) + __uint_as_float(l[i]));
                    } else {
                        tmem_ld16(taddr + (uint32_t)c0, r0);
                        tmem_ld16(taddr + (uint32_t)(NT + c0), r1);
                        tmem_ld16(taddr + (uint32_t)(2 * NT + c0), r2);
                        tmem_ld_wait();
                    }
                    if (c0 + 16 >= NT) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty[ab]);
                    }
                    // L3: rows 4t .. 4t+3 are read by layer-3 tile 0 (t <= 3) and tile 1 (t >= 3) of the previous patch
                    if (L3 && c0 == 0) RP_WAIT(1, mbar_wait(&f3_empty[t < 3 ? 0 : 1], (k & 1) ^ 1));
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        const float left = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[i]), 1);
                        const float right = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[i]), 1);
                        const float acc = fmaf(left, mask_l, fmaf(right, mask_r, __uint_as_float(r1[i])));   // 0/1 masks: zero padding outside the row
                        v[i] = fmaxf(fmaf(acc, a.inv_scale, L3 ? s_bias[c0 + i] : bias2[c0 + i]), 0.f);   // L3: from shared memory (registers spill at 25 warps)
                    }
#pragma unroll
                    for (int g = 0; g < 2; g++) {
                        uint4 hi, lo;
                        split_pack8<OSA, BF>(v + g * 8, hi, lo);
                        if (L3) {   // layer-3 input groups: hi, then lo
                            *reinterpret_cast<uint4*>(obase + (size_t)(c0 / 8 + g) * GS3 * 16) = hi;
                            *reinterpret_cast<uint4*>(obase + (size_t)(Cfg::KC3 + c0 / 8 + g) * GS3 * 16) = lo;
                            continue;
                        }
                        const size_t goff = (size_t)(c0 / 8 + g) * 1024 * 16;
                        *reinterpret_cast<uint4*>(obase + goff) = hi;
                        if (OSA == 1) *reinterpret_cast<uint4*>(obase + (size_t)(COUT / 8) * 1024 * 16 + goff) = lo;
                        if (OSA == 2) *reinterpret_cast<uint2*>(outp + Cfg::HI_OUT_BYTES + ((size_t)(c0 / 8 + g) * 1024 + layout_slot(L_S2_16, y, x, 0)) * 8) = pack_lo8(lo);
                    }
                }
                if (L3) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    if (t <= 3) mbar_arrive(&f3_full[0]);
                    if (t >= 3) mbar_arrive(&f3_full[1]);
                }
            }
        }
        if (warp == Cfg::W_L2) XP_STORE(0, 1);
    } else if (warp >= Cfg::W_L1 && warp < Cfg::W_MMA) {
        // ===== layer-1 epilogue: TMEM -> bias + ReLU -> fp16 (hi [+lo]) -> shared-memory stage of layer 2 =====
        const int q = warp & 3;
        int it = 0, c1cnt = 0;
        float bias1[C1];   // registers: a shared-memory read per use would cost the shared-memory pipe 16 wavefronts per tile and warp
#pragma unroll
        for (int i = 0; i < C1; i++) bias1[i] = s_bias1[i];
        RP_DECL;
        for (int pi = next_valid(blockIdx.x); pi < a.n; pi = next_valid(pi + gridDim.x), it++) {
            const int s = L3 ? 0 : (it & 1);
            if (!L3) RP_WAIT(0, mbar_wait(&empty[s], ((it >> 1) & 1) ^ 1));
            unsigned char* st = sIn + (size_t)s * Cfg::SLOT_STAGE * 16;
#pragma unroll 1
            for (int t = 0; t < TILES; t++, c1cnt++) {
                const int b = c1cnt % NL1;
                RP_WAIT(1, mbar_wait(&c1_full[b], (c1cnt / NL1) & 1));
                tc_fence_after();
                const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * Cfg::ACC1);
                uint32_t r[32];
                tmem_ld32(taddr, r);
                tmem_ld_wait();
                if (Cfg::S1) {   // [x*w_hi | x_hi*w_lo] side by side: add the halves
#pragma unroll
                    for (int i = 0; i < 16; i++) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r[16 + i]));
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&c1_empty[b]);
                if (L3) RP_WAIT(0, mbar_wait(&empty[t], (it & 1) ^ 1));   // the previous patch's layer-2 MMAs are done with stage tile t
                const int slot = t * 128 + q * 32 + lane + 32;      // pixel m = t*128 + row sits one (zero) row into the stage
#pragma unroll
                for (int g = 0; g < C1 / 8; g++) {
                    float v[8];
#pragma unroll
                    for (int e = 0; e < 8; e++) v[e] = fmaxf(fmaf(__uint_as_float(r[g * 8 + e]), src.w1_inv, bias1[g * 8 + e]), 0.f);
                    uint4 hi, lo;
                    split_pack8<SA, BF>(v, hi, lo);
                    *reinterpret_cast<uint4*>(st + ((size_t)g * GS + slot) * 16) = hi;
                    if (SA) *reinterpret_cast<uint4*>(st + ((size_t)(KC + g) * GS + slot) * 16) = lo;
                }
                if (L3) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_arrive(&full[t]);
                }
            }
            if (!L3) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_arrive(&full[s]);
            }
        }
        if (warp == Cfg::W_L1) XP_STORE(0, 2);
    } else if (L3 && warp >= Cfg::W_L3 && warp < Cfg::W_L2) {
        // ===== layer-3 epilogue (tcx_conv's stride-2 arithmetic): TMEM -> x shift -> bias + ReLU -> fp16 hi + lo -> global (L_S1_16) =====
        constexpr int W3 = In3::W;
        const int q = warp & 3;
        const int r = q * 32 + lane;
        int k = 0;
        RP_DECL;
        for (int pi = next_valid(blockIdx.x); pi < a.n; pi = next_valid(pi + gridDim.x), k++) {
            unsigned char* outp = reinterpret_cast<unsigned char*>(a3.out) + (size_t)pi * Cfg::UNIT_OUT3_BYTES;
#pragma unroll 1
            for (int u = 0; u < In3::TILES; u++) {
                RP_WAIT(0, mbar_wait(&t3_full[u], k & 1));
                tc_fence_after();
                const int m = u * 128 + r, y = m / W3, x = m - y * W3;
                const float mask_l = x > 0 ? 1.f : 0.f;
                const uint32_t taddr = tmem_l3 + ((uint32_t)(q * 32) << 16) + (uint32_t)(u * Cfg::ACCW3);
                unsigned char* obase = outp + (size_t)layout_slot(L_S1_16, y, x, 0) * 16;
                constexpr size_t lo_off = (size_t)(NT3 / 8) * 256 * 16;
#pragma unroll 1
                for (int c0 = 0; c0 < NT3; c0 += 16) {
                    uint32_t r0[16], r1[16], r2[16];
                    tmem_ld16(taddr + (uint32_t)c0, r0);                   // odd plane dx0
                    tmem_ld16(taddr + (uint32_t)(NT3 + c0), r1);           // odd plane dx2
                    tmem_ld16(taddr + (uint32_t)(2 * NT3 + c0), r2);       // even plane dx1
                    tmem_ld_wait();
                    if (c0 + 16 >= NT3) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&t3_empty[u]);
                    }
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        const float left = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[i]), 1, W3);
                        const float acc = fmaf(left, mask_l, __uint_as_float(r1[i]) + __uint_as_float(r2[i]));
                        v[i] = fmaxf(fmaf(acc, a3.inv_scale, s_bias3[c0 + i]), 0.f);
                    }
#pragma unroll
                    for (int g = 0; g < 2; g++) {
                        const size_t goff = (size_t)(c0 / 8 + g) * 256 * 16;
                        uint4 hi, lo;
                        split_pack8<1, BF>(v + g * 8, hi, lo);
                        *reinterpret_cast<uint4*>(obase + goff) = hi;
                        *reinterpret_cast<uint4*>(obase + lo_off + goff) = lo;
                    }
                }
            }
        }
        if (warp == Cfg::W_L3) XP_STORE(2, 1);
    } else if (warp < 8) {
        // ===== producers (8 warps): sampler (or patch load) -> input_norm -> sliding-window planes P_hi / P_lo =====
        const int pw = warp;                                 // 0..7
        const int pt = pw * 32 + lane;                       // 0..255
        float tp[4][4], fx[4], fy[4];
        // pixel k of this thread: warp pw owns image rows 4pw .. 4pw+3; k = 8-column block, lane = (row, column) inside the 4x8 block
        auto pix_of = [&](int k) -> int { return (pw * 4 + (lane >> 3)) * 32 + k * 8 + (lane & 7); };
        auto issue_fetch = [&](int pi) {
            if (src.patches != nullptr) {
                const float* pp = src.patches + (size_t)pi * 1024;
#pragma unroll
                for (int k = 0; k < 4; k++) { tp[k][0] = pp[pix_of(k)]; tp[k][1] = tp[k][2] = tp[k][3] = 0.f; fx[k] = 0.f; fy[k] = 0.f; }
            } else {
                const int b = pi / src.cap;
                const int o = min(max(src.oct[pi], 0), src.geom.n_octaves - 1), l = min(max(src.lvl[pi], 0), src.geom.n_levels - 1);
                const int h = src.geom.h[o], w = src.geom.w[o];
                const float* img = src.pyr + src.geom.off[o][l] + (size_t)b * h * w;
                const float* Lf = src.lafs + (size_t)pi * 6;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int p = pix_of(k);
                    float px, py;
                    laf_sample_xy(Lf, h, w, p >> 5, p & 31, 1.0f / 32.0f, px, py);
                    bilinear_taps(img, h, w, px, py, tp[k], fx[k], fy[k]);
                }
            }
        };
        int pi = next_valid(blockIdx.x);
        if (pi < a.n) issue_fetch(pi);
        int it = 0;
        RP_DECL;
        while (pi < a.n) {
            float* sx = s_x + (it & 1) * SX;
            float* red = s_red + (it & 1) * 16;
            float v[4];
#pragma unroll
            for (int k = 0; k < 4; k++) v[k] = bilinear_combine(tp[k], fx[k], fy[k]);
            const int pn = next_valid(pi + gridDim.x);
            if (pn < a.n) issue_fetch(pn);
            // input_norm: mean, unbiased std + 1e-7 (two passes, as the reference)
            float sm = (v[0] + v[1]) + (v[2] + v[3]);
            for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
            if (lane == 0) red[pw * 2] = sm;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            const float mean = (((red[0] + red[2]) + (red[4] + red[6])) + ((red[8] + red[10]) + (red[12] + red[14]))) / 1024.f;
            float qs = 0.f;
#pragma unroll
            for (int k = 0; k < 4; k++) { const float d = v[k] - mean; qs = fmaf(d, d, qs); }
            for (int o = 16; o > 0; o >>= 1) qs += __shfl_xor_sync(0xffffffffu, qs, o);
            if (lane == 0) red[pw * 2 + 1] = qs;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            const float inv = 1.f / (sqrtf((((red[1] + red[3]) + (red[5] + red[7])) + ((red[9] + red[11]) + (red[13] + red[15]))) / 1023.f) + 1e-7f);
#pragma unroll
            for (int k = 0; k < 4; k++) { const int p = pix_of(k); sx[((p >> 5) + 1) * 34 + (p & 31) + 1] = (v[k] - mean) * inv; }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            // P planes, half by half
#pragma unroll 1
            for (int hh = 0; hh < 2; hh++) {
                RP_WAIT(0, mbar_wait(&p_empty[hh], (it & 1) ^ 1));   // layer-1 MMAs of the previous patch have consumed this half
                unsigned char* ph = sP + (size_t)hh * 2 * NPIXP * 16;
                // one 16-byte window per thread and step: consecutive lanes read consecutive pixels and write consecutive slots (no bank
                // conflicts; the shared-memory pipe is this kernel's busiest unit)
#pragma unroll 1
                for (int s0 = pt; s0 < NPIXP; s0 += 256) {
                    const float* rowp = sx + (hh * 16 + (s0 >> 5)) * 34 + (s0 & 31);
                    float xv[8];
#pragma unroll
                    for (int e = 0; e < 4; e++) { xv[e] = rowp[e]; xv[4 + e] = rowp[34 + e]; }
                    uint4 hi, lo;
                    split_pack8<1, BF>(xv, hi, lo);
                    *reinterpret_cast<uint4*>(ph + (size_t)s0 * 16) = hi;
                    *reinterpret_cast<uint4*>(ph + (size_t)(NPIXP + s0) * 16) = lo;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_arrive(&p_full[hh]);
            }
            it++;
            pi = pn;
        }
        if (warp == 0) XP_STORE(0, 3);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == Cfg::W_MMA) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
    }
}

}  // namespace tcx
}  // namespace ag
