// Second-generation tensor-core engine of AffNet / OriNet / HardNet (tcx_first.cuh, tcx_conv.cuh): row tiles without x padding, the
// three taps of a kernel row stacked along N, x shifts by warp shuffles in the epilogue.  Replaces the conv stacks of
// architectures.py:207-235 / 36-82 and HardNet.py:67-101 (BatchNorm folded, ReLU fused); the 8x8 heads are the GEMM kernels of
// tc_head.cuh (tc_head_kernel, tc_headx_kernel).  Per net:  tcx_first_kernel (sampler + input_norm + conv1 + conv2)  ->  tcx_conv_kernel x4;
// AffNet / OriNet: conv3 inside tcx_first_kernel as well (AG_FUSE_L3), then tcx_conv_kernel x3.
// Numerics: AffNet / OriNet with fp16 residual planes of weights and activations in every layer (three MMAs per K step, fp32-grade);
// HardNet fp16 activations, weights with their fp16 residual in layers 2 and 3 (emulation on the 2000 graf patches: plain fp16 weights give a
// descriptor error of 1.1e-3, dominated by the weight rounding of the early layers; measured on the GPU with the residuals of layers 2-3:
// <= 4.9e-4 end to end over every parity configuration; adding layer 4's residual buys 0.5e-4 for 0.29 ms per step, layer 3's is free: HBM bound).
#include <stdlib.h>
#include <string.h>

#include <vector>

#include <cuda_bf16.h>

#include "net_impl.cuh"
#include "tc_head.cuh"
#include "tcx_conv.cuh"
#include "tcx_first.cuh"

namespace ag {
namespace tcx {

static int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

static int ensure_smem_attr(const void* func, int bytes, bool* configured, const char* what) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (configured[dev]) return AG_OK;
    int rc = check_cuda(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes), what);
    if (rc == AG_OK) configured[dev] = true;
    return rc;
}

template <int CIN, int COUT, int H, int STRIDE, int NSPLIT, int STAGES, int OUT, int SA, int SW, int OSA, int EW, int BF = 0, int MC = 0>
static int launch_conv(const void* in, void* out, const __half* w, const float* b, float inv_scale, int n, int group, const int* count, cudaStream_t st) {
    constexpr int prof_id = (H == 32) ? 2 : (H == 16 ? (STRIDE == 1 ? 3 : 4) : 5);
    using Cfg = XCfg<CIN, COUT, H, STRIDE, NSPLIT, STAGES, OUT, SA, SW, OSA, EW>;
    auto kern = tcx_conv_kernel<CIN, COUT, H, STRIDE, NSPLIT, STAGES, OUT, SA, SW, OSA, EW, BF, MC>;
    static bool configured[64] = {};   // per device (the attribute is per device)
    int rc = ensure_smem_attr((const void*)kern, (int)Cfg::SMEM, configured, "tcx_conv smem attr");
    if (rc != AG_OK) return rc;
    XArgs a;
    a.in = (const __half*)in; a.out = out; a.wpk = w; a.bias = b; a.inv_scale = inv_scale; a.n = n; a.group = group; a.count = count; a.prof_id = prof_id;
    const int units = Cfg::In::PAIR ? (n + 1) / 2 : n;
    int gx = num_sms() / NSPLIT;
    if (gx > units) gx = units;
    if (gx < 1) gx = 1;
    if (MC) {   // the two channel-split CTAs of a unit as one thread-block cluster (1 x 2)
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(gx, NSPLIT); cfg.blockDim = dim3(Cfg::THREADS); cfg.dynamicSmemBytes = Cfg::SMEM; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 2; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        rc = check_cuda(cudaLaunchKernelEx(&cfg, kern, a), "tcx_conv cluster launch");
        if (rc != AG_OK) return rc;
    } else
        kern<<<dim3(gx, NSPLIT), Cfg::THREADS, Cfg::SMEM, st>>>(a);
    AG_CHECK_LAUNCH("tcx_conv_kernel");
    return AG_OK;
}

// L3 = 1: conv layer 3 fused (its weights / bias / scale in w3 / b3 / inv_scale3); it writes out3 and `out` is not used
template <int C1, int COUT, int SA, int SW, int OSA, int BF = 0, int L3 = 0>
static int launch_first(void* out, const __half* w, const float* b, float inv_scale, int n, int group, const int* count, cudaStream_t st, const FirstSrc& src,
                        void* out3 = nullptr, const __half* w3 = nullptr, const float* b3 = nullptr, float inv_scale3 = 0.f) {
    using Cfg = XFirstCfg<C1, COUT, SA, SW, OSA, L3>;
    auto kern = tcx_first_kernel<C1, COUT, SA, SW, OSA, BF, L3>;
    static bool configured[64] = {};
    int rc = ensure_smem_attr((const void*)kern, (int)Cfg::SMEM, configured, "tcx_first smem attr");
    if (rc != AG_OK) return rc;
    XArgs a;
    a.in = nullptr; a.out = out; a.wpk = w; a.bias = b; a.inv_scale = inv_scale; a.n = n; a.group = group; a.count = count; a.prof_id = 0;
    XArgs a3 = a;
    a3.out = out3; a3.wpk = w3; a3.bias = b3; a3.inv_scale = inv_scale3;
    int gx = num_sms();
    if (gx > n) gx = n;
    if (gx < 1) gx = 1;
    kern<<<gx, Cfg::THREADS, Cfg::SMEM, st>>>(a, src, a3);
    AG_CHECK_LAUNCH("tcx_first_kernel");
    return AG_OK;
}

// debug / test helper: an activation buffer in one of the HBM layouts -> fp32 [n][C][H][H] (hi + lo planes added)
__global__ void tcx_decode_kernel(const __half* __restrict__ buf, int layout, int C, int osa, int H, int n, float* __restrict__ out) {
    const size_t total = (size_t)n * C * H * H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % H), y = (int)((i / H) % H), c = (int)((i / ((size_t)H * H)) % C), pi = (int)(i / ((size_t)H * H * C));
        const int slots = layout_slots(layout);
        const size_t unit_halfs = (size_t)(C / 8) * slots * 8 * (osa == 1 ? 2 : 1) + (osa == 2 ? (size_t)(C / 8) * slots * 4 : 0);
        const int unit = layout_pair(layout) ? (pi >> 1) : pi;
        const int slot = layout_slot(layout, y, x, pi & 1);
        const __half* ub = buf + (size_t)unit * unit_halfs;
        float v = __half2float(ub[((size_t)(c / 8) * slots + slot) * 8 + (c & 7)]);
        if (osa == 1) v += __half2float(ub[((size_t)(C / 8 + c / 8) * slots + slot) * 8 + (c & 7)]);
        if (osa == 2) {   // byte residual planes behind the hi planes
            const unsigned char* lb = reinterpret_cast<const unsigned char*>(ub) + (size_t)(C / 8) * slots * 16;
            const unsigned short bits = (unsigned short)(lb[((size_t)(c / 8) * slots + slot) * 8 + (c & 7)] << 8);
            v += __half2float(__ushort_as_half(bits));
        }
        out[i] = v;
    }
}

}  // namespace tcx

// ---- sources of the first kernel: materialised patches, or the pyramid + keypoints ---------------------------------------------------
tc::FirstSrc tc_src_patches(const float* patches) {
    tc::FirstSrc s;
    memset(&s, 0, sizeof(s));
    s.patches = patches;
    s.cap = 1;
    return s;
}

tc::FirstSrc tc_src_pyramid(const ag_pyramid_plan_t* p, const float* pyr, const float* lafs, const int* oct, const int* lvl, int cap) {
    tc::FirstSrc s;
    memset(&s, 0, sizeof(s));
    s.pyr = pyr; s.lafs = lafs; s.oct = oct; s.lvl = lvl; s.cap = cap;
    s.geom.n_octaves = p->n_octaves; s.geom.n_levels = p->n_levels;
    for (int o = 0; o < AG_MAX_OCTAVES; o++) {
        s.geom.h[o] = p->h[o]; s.geom.w[o] = p->w[o];
        for (int l = 0; l < AG_MAX_LEVELS; l++) s.geom.off[o][l] = p->level_offset[o][l];
    }
    return s;
}

// ---- heads ----------------------------------------------------------------------------------------------------------------------------
// HardNet 8x8 head GEMM + BatchNorm + L2 norm over the head operand a trunk left in `headbuf`
int tc_hardnet_head(const ag_net* net, const void* headbuf, int n, int group, const int* count, float* out, cudaStream_t st, int bf16) {
    using namespace tc;
    static SmemAttrOnce once0, once1;
    {
        int rc = once0.ensure(tc_head_kernel<0>, HEAD_SMEM, "tc_head smem attr");
        if (rc == AG_OK) rc = once1.ensure(tc_head_kernel<1>, HEAD_SMEM, "tc_head smem attr");
        if (rc != AG_OK) return rc;
    }
    if (bf16) tc_head_kernel<1><<<(n + 127) / 128, 192, HEAD_SMEM, st>>>((const __half*)headbuf, net->d_headh_bf, net->d_head_b, out, n, group, count);
    else tc_head_kernel<0><<<(n + 127) / 128, 192, HEAD_SMEM, st>>>((const __half*)headbuf, net->d_headh, net->d_head_b, out, n, group, count);
    AG_CHECK_LAUNCH("tc_head_kernel");
    return AG_OK;
}

// AffNet / OriNet head on tensor cores over the hi/lo feature planes the trunk leaves in `feat`
int tc_headx_forward(const ag_net* net, const void* feat, int n, int group, const int* count, float* out, float* angle, cudaStream_t st, float* raw) {
    using namespace tc;
    static SmemAttrOnce once0, once1;
    {
        int rc = once0.ensure(tc_headx_kernel<0>, HX_SMEM, "tc_headx smem attr");
        if (rc == AG_OK) rc = once1.ensure(tc_headx_kernel<1>, HX_SMEM, "tc_headx smem attr");
        if (rc != AG_OK) return rc;
    }
    const int tiles = (n + 127) / 128;
    if (net->kind == AG_NET_AFFNET) tc_headx_kernel<0><<<tiles, 192, HX_SMEM, st>>>((const __half*)feat, net->d_headh, net->d_head_b, net->head_inv_scale, out, nullptr, raw, n, group, count);
    else tc_headx_kernel<1><<<tiles, 192, HX_SMEM, st>>>((const __half*)feat, net->d_headh, net->d_head_b, net->head_inv_scale, out, angle, raw, n, group, count);
    AG_CHECK_LAUNCH("tc_headx_kernel");
    return AG_OK;
}

// bytes of the head-GEMM operand of n patches (hi + lo planes, padded to whole 128-patch tiles)
size_t tc_headx_bytes(int n) { return (size_t)((n + 127) / 128) * 2 * tc::HX_PLANE_TILE; }

// ---- weight packing (host) --------------------------------------------------------------------------------------------------------
// wf: fp32 [tap = dy*3+dx][ci][co] (BatchNorm folded), scale: power of two.  Blocks per (split, dy, 16 input channels):
//   stride 1: [K group (2)][part hi|lo][dx 0,1,2][co][8]
//   stride 2: odd-x plane [K group][part][dx 0,2][co][8], then even-x plane [K group][part][dx 1][co][8]
static __half bf16_bits_as_half(float v) {   // bf16(v) stored in a 16-bit slot of the (type-agnostic) weight buffer
    const __nv_bfloat16 b = __float2bfloat16_rn(v);
    __half h;
    memcpy(&h, &b, 2);
    return h;
}
static float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

void tcx_pack_layer(const float* wf, int ci, int co, int stride, int nsplit, int sw, float scale, std::vector<__half>& out, int bf16) {
    const int nt = co / nsplit;
    auto put = [&](int dy, int dx, int cin, int c, int part) {
        const float v = scale * wf[((size_t)(dy * 3 + dx) * ci + cin) * co + c];
        if (bf16) {
            const float hi = bf16_round(v);
            out.push_back(bf16_bits_as_half(part == 0 ? hi : v - hi));
        } else {
            const __half hi = __float2half_rn(v);
            out.push_back(part == 0 ? hi : __float2half_rn(v - __half2float(hi)));
        }
    };
    for (int sp = 0; sp < nsplit; sp++)
        for (int dy = 0; dy < 3; dy++)
            for (int j = 0; j < ci / 16; j++) {
                if (stride == 1) {
                    for (int kg = 0; kg < 2; kg++)
                        for (int part = 0; part <= sw; part++)
                            for (int dx = 0; dx < 3; dx++)
                                for (int c = 0; c < nt; c++)
                                    for (int e = 0; e < 8; e++) put(dy, dx, (2 * j + kg) * 8 + e, sp * nt + c, part);
                } else {
                    for (int kg = 0; kg < 2; kg++)
                        for (int part = 0; part <= sw; part++)
                            for (int dx = 0; dx < 3; dx += 2)
                                for (int c = 0; c < nt; c++)
                                    for (int e = 0; e < 8; e++) put(dy, dx, (2 * j + kg) * 8 + e, sp * nt + c, part);
                    for (int kg = 0; kg < 2; kg++)
                        for (int part = 0; part <= sw; part++)
                            for (int c = 0; c < nt; c++)
                                for (int e = 0; e < 8; e++) put(dy, 1, (2 * j + kg) * 8 + e, sp * nt + c, part);
                }
            }
}

int tcx_nsplit(int kind, int layer) { return (kind == AG_NET_HARDNET && layer >= 4) ? 2 : 1; }
// weight residual copies: AffNet / OriNet every layer; HardNet layers 2-3 (layer index 1..2; see the A/B switches)
#ifndef AG_HARD_SW2
#define AG_HARD_SW2 1
#endif
#ifndef AG_HARD_SW3
#define AG_HARD_SW3 1   // HardNet layer 3 / layer 4 weight residuals (A/B switches for the accuracy / time trade, see DESIGN.md)
#endif
#ifndef AG_HARD_SW4
#define AG_HARD_SW4 0   // measured r02: without it the worst descriptor error over all parity configurations is 4.9e-4 (with: 4.4e-4) and layer 4 is 0.29 ms per step faster
#endif
int tcx_split_w(int kind, int layer) { return kind == AG_NET_HARDNET ? (layer == 1 ? AG_HARD_SW2 : layer == 2 ? AG_HARD_SW3 : layer == 3 ? AG_HARD_SW4 : 0) : 1; }
int tcx_stride(int layer) { return (layer == 2 || layer == 4) ? 2 : 1; }

// bytes of each of the two ping-pong activation buffers for n patches (largest layer output: 64 KiB per patch; pair layouts round n up)
size_t tcx_act_bytes(int n) { return (size_t)(n + 1) * 65536; }

// ---- trunks -------------------------------------------------------------------------------------------------------------------------
// AffNet / OriNet (same shapes, own weights): features as fp16 hi + lo planes in the head-GEMM layout.  upto: stop after conv layer
// `upto` (2..6; for the debug decode), 6 = whole trunk.
// epilogue warps of AffNet / OriNet layers 3 and 4 (4 | 8)
// cluster-multicast input of HardNet's channel-split layers: layer 5 0.38 -> 0.35 ms, layer 6 unchanged (kept off)
#ifndef AG_HARD_MC5
#define AG_HARD_MC5 1
#endif
#ifndef AG_HARD_MC6
#define AG_HARD_MC6 0
#endif
#ifndef AG_HARD_EW4
#define AG_HARD_EW4 16   // HardNet layer 4 (N = 192, two accumulator buffers): 16 epilogue warps = 2 tile sets x 2 column halves, 0.56 -> 0.49 ms
#endif
#ifndef AG_AFF_EW6
#define AG_AFF_EW6 8
#endif
// Residual planes of layer 2's output (the largest activation, read by the HBM-bound layer 3) as bytes (1) or fp16 (0).  Measured
// (tests/test_gpu_tcx.py, bench A/B): with byte planes AffNet's A stays at 4.5e-6 of the oracle and layer 3 goes from 0.80 to 0.69 ms per
// step (the same in front of layer 5 made that layer slower, 0.37 -> 0.41 ms: not wired).  OFF by default: the application test with the
// hand-crafted orientation (test_graf_1_to_6_application_counts[hcori]) then has one keypoint of 2996 whose frame differs from the
// oracle's by more than its near-tie accounting allows (a pixel on a histogram-bin boundary, DESIGN.md section 8; the accounting would
// have to cover that case before the switch can be on).  OriNet's angle error grows from
// 3e-5 to 1.2e-4 rad with byte planes (its atan2 amplifies): off for OriNet as well.
#ifndef AG_AFF_LO8
#define AG_AFF_LO8 0
#endif
#ifndef AG_ORI_LO8
#define AG_ORI_LO8 0
#endif
static inline int tcx_lox(const ag_net* net) { return ((net->kind == AG_NET_AFFNET) ? AG_AFF_LO8 : AG_ORI_LO8) ? 2 : 1; }
#ifndef AG_AFF_EW3
#define AG_AFF_EW3 4
#endif
#ifndef AG_AFF_EW4
#define AG_AFF_EW4 8   // layer 4 waited for its 4-warp epilogue 23 % of the time: 0.72 -> 0.61 ms (AffNet), 0.48 -> 0.41 (OriNet); layer 3 is HBM bound (no change)
#endif
// Conv layer 3 fused into the first kernel (tcx_first.cuh, L3 = 1): layer 2's output stays in shared memory instead of a 64 KiB per
// patch round trip through HBM, and the step has one launch fewer per net.  Bit-identical to the unfused pair (tests/test_gpu_fused_l3.py).
// AG_FUSE_L3=0 builds with the unfused pair as the default; ag_debug_fuse_l3() switches at run time.  The byte residual planes
// (AG_AFF_LO8 / AG_ORI_LO8) only exist to shrink that HBM round trip: a net built with them runs the unfused pair.
#ifndef AG_FUSE_L3
#define AG_FUSE_L3 1
#endif
static int g_tcx_fuse_l3 = AG_FUSE_L3;
template <int LOX>
static int trunk_affori_t(const ag_net* net, const tc::FirstSrc& src0, int n, int group, const int* count, void* bufA, void* bufB, void* feat,
                          cudaStream_t st, int upto) {
    using namespace tcx;
    tc::FirstSrc src = src0;
    src.w1 = net->d_w1; src.b1 = net->d_b[0]; src.w1_inv = net->w_inv_scale[0]; src.w1_scale = 1.0f / net->w_inv_scale[0];
    int rc;
    if (LOX == 1 && g_tcx_fuse_l3 && upto >= 3) {   // layer 2's output only exists on the unfused path (upto = 2)
        if ((rc = launch_first<16, 16, 1, 1, 1, 0, 1>(nullptr, net->d_wx[1], net->d_b[1], net->w_inv_scale[1], n, group, count, st, src, bufA, net->d_wx[2],
                                                      net->d_b[2], net->w_inv_scale[2])))
            return rc;
    } else {
        if ((rc = launch_first<16, 16, 1, 1, LOX>(bufB, net->d_wx[1], net->d_b[1], net->w_inv_scale[1], n, group, count, st, src))) return rc;
        if (upto <= 2) return AG_OK;
        if ((rc = launch_conv<16, 32, 32, 2, 1, 3, L_S1_16, LOX, 1, 1, AG_AFF_EW3>(bufB, bufA, net->d_wx[2], net->d_b[2], net->w_inv_scale[2], n, group, count, st))) return rc;
    }
    if (upto <= 3) return AG_OK;
    if ((rc = launch_conv<32, 32, 16, 1, 1, 4, L_S2_8P, 1, 1, 1, AG_AFF_EW4>(bufA, bufB, net->d_wx[3], net->d_b[3], net->w_inv_scale[3], n, group, count, st))) return rc;
    if (upto <= 4) return AG_OK;
    if ((rc = launch_conv<32, 64, 16, 2, 1, 2, L_S1_8P, 1, 1, 1, 8>(bufB, bufA, net->d_wx[4], net->d_b[4], net->w_inv_scale[4], n, group, count, st))) return rc;
    if (upto <= 5) return AG_OK;
    return launch_conv<64, 64, 8, 1, 1, 2, L_HEAD, 1, 1, 1, AG_AFF_EW6>(bufA, feat, net->d_wx[5], net->d_b[5], net->w_inv_scale[5], n, group, count, st);
}
int tcx_trunk_affori(const ag_net* net, const tc::FirstSrc& src0, int n, int group, const int* count, void* bufA, void* bufB, void* feat,
                     cudaStream_t st, int upto) {
    return tcx_lox(net) == 2 ? trunk_affori_t<2>(net, src0, n, group, count, bufA, bufB, feat, st, upto)
                             : trunk_affori_t<1>(net, src0, n, group, count, bufA, bufB, feat, st, upto);
}

template <int BF>
static int trunk_hardnet_t(const ag_net* net, const tc::FirstSrc& src0, int n, int group, const int* count, void* bufA, void* bufB, void* headbuf,
                           cudaStream_t st, int upto) {
    using namespace tcx;
    tc::FirstSrc src = src0;
    src.w1 = net->d_w1; src.b1 = net->d_b[0]; src.w1_inv = net->w_inv_scale[0]; src.w1_scale = 1.0f / net->w_inv_scale[0];
    __half* const* wx = BF ? net->d_wx_bf : net->d_wx;
    int rc;
    if ((rc = launch_first<32, 32, 0, AG_HARD_SW2, 0, BF>(bufB, wx[1], net->d_b[1], net->w_inv_scale[1], n, group, count, st, src))) return rc;
    if (upto <= 2) return AG_OK;
    if ((rc = launch_conv<32, 64, 32, 2, 1, 2, L_S1_16, 0, AG_HARD_SW3, 0, 8, BF>(bufB, bufA, wx[2], net->d_b[2], net->w_inv_scale[2], n, group, count, st))) return rc;
    if (upto <= 3) return AG_OK;
    if ((rc = launch_conv<64, 64, 16, 1, 1, 2, L_S2_8P, 0, AG_HARD_SW4, 0, AG_HARD_EW4, BF>(bufA, bufB, wx[3], net->d_b[3], net->w_inv_scale[3], n, group, count, st))) return rc;
    if (upto <= 4) return AG_OK;
    if ((rc = launch_conv<64, 128, 16, 2, 2, 2, L_S1_8P, 0, 0, 0, 8, BF, AG_HARD_MC5>(bufB, bufA, wx[4], net->d_b[4], net->w_inv_scale[4], n, group, count, st))) return rc;
    if (upto <= 5) return AG_OK;
    return launch_conv<128, 128, 8, 1, 2, 2, L_HEAD, 0, 0, 0, 8, BF, AG_HARD_MC6>(bufA, headbuf, wx[5], net->d_b[5], net->w_inv_scale[5], n, group, count, st);
}

int tcx_trunk_hardnet(const ag_net* net, const tc::FirstSrc& src0, int n, int group, const int* count, void* bufA, void* bufB, void* headbuf,
                      cudaStream_t st, int upto, int bf16) {
    return bf16 ? trunk_hardnet_t<1>(net, src0, n, group, count, bufA, bufB, headbuf, st, upto)
                : trunk_hardnet_t<0>(net, src0, n, group, count, bufA, bufB, headbuf, st, upto);
}

}  // namespace ag

using namespace ag;

extern "C" {

// Developer diagnostic (tests/test_gpu_tcx.py): run the second-generation trunk of `net` on materialised patches [n,32,32] up to conv
// layer `upto` (2..5) and decode that layer's output (fp16 hi [+ lo] planes in its HBM layout) to fp32 [n][C][H][H].
int ag_debug_tcx_layer(const ag_net_t* net, const float* d_patches, int n, int upto, float* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(net && d_patches && d_out && d_ws, "NULL argument");
    AG_REQUIRE(upto >= 2 && upto <= 5 && n >= 1, "layer out of range");
    const size_t act = align_up(tcx_act_bytes(n), 256);
    AG_REQUIRE(ws_bytes >= 2 * act, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)d_ws;
    const tc::FirstSrc src = tc_src_patches(d_patches);
    const bool hard = net->kind == AG_NET_HARDNET;
    int rc = hard ? tcx_trunk_hardnet(net, src, n, n, nullptr, base, base + act, nullptr, st, upto)
                  : tcx_trunk_affori(net, src, n, n, nullptr, base, base + act, nullptr, st, upto);
    if (rc) return rc;
    // layer l (2..5) writes: 2 -> bufB (L_S2_16, 32x32), 3 -> bufA (L_S1_16, 16x16), 4 -> bufB (L_S2_8P, 16x16), 5 -> bufA (L_S1_8P, 8x8)
    const int lay = upto == 2 ? tcx::L_S2_16 : upto == 3 ? tcx::L_S1_16 : upto == 4 ? tcx::L_S2_8P : tcx::L_S1_8P;
    const int H = upto == 2 ? 32 : (upto <= 4 ? 16 : 8);
    const int Cb = hard ? 32 : 16;
    const int C = upto == 2 ? Cb : (upto <= 4 ? 2 * Cb : 4 * Cb);
    const void* buf = (upto == 2 || upto == 4) ? base + act : base;
    // the planes layer 2 writes carry byte residuals when the net uses them (tcx_lox)
    const int osa = hard ? 0 : (upto == 2 ? tcx_lox(net) : 1);
    tcx::tcx_decode_kernel<<<296, 256, 0, st>>>((const __half*)buf, lay, C, osa, H, n, d_out);
    AG_CHECK_LAUNCH("tcx_decode_kernel");
    return AG_OK;
}

// Developer switch: 1 = conv layer 3 of AffNet / OriNet fused into the first kernel (default unless built with AG_FUSE_L3=0), 0 = the
// unfused pair.  Returns the previous mode.
int ag_debug_fuse_l3(int fused) {
    const int old = g_tcx_fuse_l3;
    g_tcx_fuse_l3 = fused ? 1 : 0;
    return old;
}

}  // extern "C"

#ifdef AG_ROLE_PROF
// developer-only: per-CTA role cycle counters of the last second-generation launches (tcx_conv.cuh)
extern "C" int ag_debug_role_prof_x(unsigned long long* out) {
    if (cudaMemcpyFromSymbol(out, ag::tcx::g_xprof, sizeof(unsigned long long) * 8 * 160 * 20) != cudaSuccess) return 1;
    void* p = nullptr;
    return (cudaGetSymbolAddress(&p, ag::tcx::g_xprof) == cudaSuccess && cudaMemset(p, 0, sizeof(unsigned long long) * 8 * 160 * 20) == cudaSuccess) ? 0 : 1;
}
#endif
