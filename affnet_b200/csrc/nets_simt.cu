// AffNet / OriNet / HardNet forward, fp32 SIMT path (SURVEY.md §8a rows a9, a10, a12, a16).
//
// Replaces AffNetFast.forward (architectures.py:204-252), OriNetFast.forward (architectures.py:33-82) and
// HardNet.forward (HardNet.py:61-101) in eval mode: per-patch input normalisation, six conv3x3 + BatchNorm
// (affine=False, eps 1e-5, running stats; folded into the weights at upload) + ReLU, then the 8x8 head.
// This is the exact-fp32 engine: every layer is a direct convolution with the whole (padded) input of one
// patch staged in shared memory, activations in NCHW through L2-resident scratch.  The tensor-core engine
// (nets_tcx.cu) is the default; ag_net_create below packs the weights of both.
#include <math.h>

#include <vector>

#include <cuda_bf16.h>

#include "net_impl.cuh"

namespace ag {

constexpr float BN_EPS = 1e-5f;
constexpr int CNT = 256;

struct LayerCfg {
    int cin, cout, stride, hin;
};
static const LayerCfg kAffCfg[6] = {{1, 16, 1, 32}, {16, 16, 1, 32}, {16, 32, 2, 32}, {32, 32, 1, 16}, {32, 64, 2, 16}, {64, 64, 1, 8}};
static const LayerCfg kHardCfg[6] = {{1, 32, 1, 32}, {32, 32, 1, 32}, {32, 64, 2, 32}, {64, 64, 1, 16}, {64, 128, 2, 16}, {128, 128, 1, 8}};

}  // namespace ag

namespace ag {

// ---- direct 3x3 convolution, one patch (x cout tile) per CTA -------------------------------------------
template <int CIN, int COUT, int HIN, int STRIDE, int CT, int CK, bool NORM>
__global__ void __launch_bounds__(CNT) conv3x3_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                       const float* __restrict__ wpk, const float* __restrict__ bias,
                                                       int group, const int* __restrict__ count) {
    constexpr int HOUT = HIN / STRIDE, NP = HOUT * HOUT, PPT = 4, PT = NP / PPT, CGN = CNT / PT, CPT = CT / CGN;
    constexpr int HP = HIN + 2, WP = HIN + 2;
    static_assert(PT * CGN == CNT && CPT * CGN == CT && CPT % 4 == 0, "bad tiling");
    static_assert(CIN % CK == 0, "bad cin chunk");
    extern __shared__ float smem[];
    float* s_in = smem;                    // [CIN][HP][WP]
    float* s_w = smem + CIN * HP * WP;     // [9][CK][CT]
    __shared__ float s_red[CNT / 32][2];

    const int pi = blockIdx.x;
    if (count != nullptr && (pi % group) >= count[pi / group]) return;
    const int ct0 = blockIdx.y * CT;
    const float* src = in + (size_t)pi * CIN * HIN * HIN;

    float mean = 0.f, inv = 1.f;
    if (NORM) {
        // input_norm: (x - mean) / (std_unbiased + 1e-7)    architectures.py:231-235, HardNet.py:92-96
        float s = 0.f;
        for (int i = threadIdx.x; i < HIN * HIN; i += CNT) s += src[i];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5][0] = s;
        __syncthreads();
        s = 0.f;
        for (int i = 0; i < CNT / 32; i++) s += s_red[i][0];
        mean = s / (float)(HIN * HIN);
        float q = 0.f;
        for (int i = threadIdx.x; i < HIN * HIN; i += CNT) { const float d = src[i] - mean; q = fmaf(d, d, q); }
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5][1] = q;
        __syncthreads();
        q = 0.f;
        for (int i = 0; i < CNT / 32; i++) q += s_red[i][1];
        inv = 1.f / (sqrtf(q / (float)(HIN * HIN - 1)) + 1e-7f);
    }
    // stage the zero-padded input
    for (int i = threadIdx.x; i < CIN * HP * WP; i += CNT) {
        const int c = i / (HP * WP), r = i - c * HP * WP, y = r / WP, x = r - y * WP;
        float v = 0.f;
        if (y >= 1 && y <= HIN && x >= 1 && x <= HIN) {
            v = src[(size_t)c * HIN * HIN + (y - 1) * HIN + (x - 1)];
            if (NORM) v = (v - mean) * inv;
        }
        s_in[i] = v;
    }

    const int pt = threadIdx.x % PT, cg = threadIdx.x / PT;
    int poff[PPT];
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        const int p = pt + k * PT, y = p / HOUT, x = p - y * HOUT;
        poff[k] = (y * STRIDE) * WP + x * STRIDE;
    }
    float acc[PPT][CPT];
#pragma unroll
    for (int j = 0; j < CPT; j++) {
        const float bv = bias[ct0 + cg * CPT + j];
#pragma unroll
        for (int k = 0; k < PPT; k++) acc[k][j] = bv;
    }

    for (int c0 = 0; c0 < CIN; c0 += CK) {
        __syncthreads();  // previous chunk consumed (and input staged on the first iteration)
        for (int i = threadIdx.x; i < 9 * CK * CT; i += CNT) {
            const int tap = i / (CK * CT), r = i - tap * CK * CT, c = r / CT, co = r - c * CT;
            s_w[i] = __ldg(wpk + ((size_t)tap * CIN + c0 + c) * COUT + ct0 + co);
        }
        __syncthreads();
#pragma unroll 1
        for (int c = 0; c < CK; c++) {
            const float* ip = s_in + (c0 + c) * HP * WP;
#pragma unroll
            for (int tap = 0; tap < 9; tap++) {
                const int toff = (tap / 3) * WP + (tap % 3);
                float a[PPT];
#pragma unroll
                for (int k = 0; k < PPT; k++) a[k] = ip[poff[k] + toff];
                const float4* wp = reinterpret_cast<const float4*>(s_w + (tap * CK + c) * CT + cg * CPT);
#pragma unroll
                for (int j4 = 0; j4 < CPT / 4; j4++) {
                    const float4 wv = wp[j4];
#pragma unroll
                    for (int k = 0; k < PPT; k++) {
                        acc[k][j4 * 4 + 0] = fmaf(a[k], wv.x, acc[k][j4 * 4 + 0]);
                        acc[k][j4 * 4 + 1] = fmaf(a[k], wv.y, acc[k][j4 * 4 + 1]);
                        acc[k][j4 * 4 + 2] = fmaf(a[k], wv.z, acc[k][j4 * 4 + 2]);
                        acc[k][j4 * 4 + 3] = fmaf(a[k], wv.w, acc[k][j4 * 4 + 3]);
                    }
                }
            }
        }
    }
    float* dst = out + (size_t)pi * COUT * NP;
#pragma unroll
    for (int j = 0; j < CPT; j++)
#pragma unroll
        for (int k = 0; k < PPT; k++) dst[(size_t)(ct0 + cg * CPT + j) * NP + pt + k * PT] = fmaxf(acc[k][j], 0.f);
}

template <int CIN, int COUT, int HIN, int STRIDE, int CT, int CK, bool NORM>
static int launch_conv(const float* in, float* out, const float* w, const float* b, int n, int group, const int* count,
                       cudaStream_t st) {
    constexpr size_t smem = sizeof(float) * ((size_t)CIN * (HIN + 2) * (HIN + 2) + 9 * CK * CT);
    static SmemAttrOnce attr_once;
    auto kern = conv3x3_kernel<CIN, COUT, HIN, STRIDE, CT, CK, NORM>;
    {
        int rc = attr_once.ensure(kern, smem, "conv smem attr");
        if (rc != AG_OK) return rc;
    }
    kern<<<dim3(n, COUT / CT), CNT, smem, st>>>(in, out, w, b, group, count);
    AG_CHECK_LAUNCH("conv3x3_kernel");
    return AG_OK;
}

// ---- heads --------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// AffNet: conv8x8(64->3)+bias, tanh, A = [[1+x0, 0],[x1, 1+x2]], rectifyAffineTransformationUpIsUp (LAF.py:285-291)
__global__ void affnet_head_kernel(const float* __restrict__ feat, const float* __restrict__ w, const float* __restrict__ bias,
                                   float* __restrict__ out, int n, int group, const int* __restrict__ count) {
    const int pi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (pi >= n) return;
    if (count != nullptr && (pi % group) >= count[pi / group]) return;
    const float* f = feat + (size_t)pi * 4096;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int i = lane; i < 4096; i += 32) {
        const float v = f[i];
        s0 = fmaf(v, __ldg(w + i), s0); s1 = fmaf(v, __ldg(w + 4096 + i), s1); s2 = fmaf(v, __ldg(w + 8192 + i), s2);
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    if (lane == 0) {
        const float a00 = 1.0f + tanhf(s0 + bias[0]), a01 = 0.f, a10 = tanhf(s1 + bias[1]), a11 = 1.0f + tanhf(s2 + bias[2]);
        const float det = sqrtf(fabsf(a00 * a11 - a10 * a01 + 1e-10f));
        const float b2a2 = sqrtf(a01 * a01 + a00 * a00);
        float* o = out + (size_t)pi * 4;
        o[0] = b2a2 / det; o[1] = 0.f;
        o[2] = (a11 * a01 + a10 * a00) / (b2a2 * det); o[3] = det / b2a2;
    }
}

// OriNet: conv8x8(64->2, padding=1)+bias on the 8x8 map -> 3x3, tanh, mean, atan2, rotation (architectures.py:57-59,76-82).
// The padded 8x8 kernel sliding over an 8x8 map is 18 dot products of length 4096 against per-position shifted copies of the
// weights (w_eff[k][c*9 + oy*3 + ox], built at upload): one warp handles 4 patches, lanes stride over k, the 72 accumulators
// are reduced by shuffles; weights go through shared memory in chunks so every CTA reads them once.
constexpr int OH_P = 4, OH_W = 8, OH_KC = 256;   // patches per warp, warps per CTA, k-chunk
__global__ void __launch_bounds__(OH_W * 32) orinet_head_kernel(const float* __restrict__ feat, const float* __restrict__ weff, const float* __restrict__ bias,
                                                                 float* __restrict__ out, float* __restrict__ angle_out, int n, int group,
                                                                 const int* __restrict__ count) {
    __shared__ __align__(16) float s_w[OH_KC][20];   // 18 used, rows padded to 80 B
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p0 = (blockIdx.x * OH_W + warp) * OH_P;
    float acc[OH_P][18];
#pragma unroll
    for (int q = 0; q < OH_P; q++)
#pragma unroll
        for (int o = 0; o < 18; o++) acc[q][o] = 0.f;
    const float* f[OH_P];
#pragma unroll
    for (int q = 0; q < OH_P; q++) f[q] = feat + (size_t)min(p0 + q, n - 1) * 4096;
    for (int k0 = 0; k0 < 4096; k0 += OH_KC) {
        __syncthreads();
        for (int i = threadIdx.x; i < OH_KC * 18; i += OH_W * 32) s_w[i / 18][i % 18] = __ldg(weff + (size_t)k0 * 18 + i);
        __syncthreads();
#pragma unroll 2
        for (int kk = lane; kk < OH_KC; kk += 32) {
            float v[OH_P];
#pragma unroll
            for (int q = 0; q < OH_P; q++) v[q] = f[q][k0 + kk];
            const float4* wr = reinterpret_cast<const float4*>(&s_w[kk][0]);
            const float4 w0 = wr[0], w1 = wr[1], w2 = wr[2], w3 = wr[3];
            const float2 w4 = *reinterpret_cast<const float2*>(&s_w[kk][16]);
            const float wv[18] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w, w4.x, w4.y};
#pragma unroll
            for (int q = 0; q < OH_P; q++)
#pragma unroll
                for (int o = 0; o < 18; o++) acc[q][o] = fmaf(v[q], wv[o], acc[q][o]);
        }
    }
#pragma unroll
    for (int q = 0; q < OH_P; q++) {
        float m0 = 0.f, m1 = 0.f;
#pragma unroll
        for (int o = 0; o < 9; o++) {
            m0 += tanhf(warp_sum(acc[q][o]) + bias[0]);
            m1 += tanhf(warp_sum(acc[q][9 + o]) + bias[1]);
        }
        const int pi = p0 + q;
        if (lane != 0 || pi >= n) continue;
        if (count != nullptr && (pi % group) >= count[pi / group]) continue;
        m0 /= 9.0f; m1 /= 9.0f;
        const float ang = atan2f(m0 + 1e-8f, m1 + 1e-8f);  // architectures.py:78
        if (angle_out) angle_out[pi] = ang;
        if (out) {
            const float c = cosf(ang), sn = sinf(ang);  // get_rotation_matrix, LAF.py:276-283
            float* o = out + (size_t)pi * 4;
            o[0] = c; o[1] = sn; o[2] = -sn; o[3] = c;
        }
    }
}

// HardNet: conv8x8(128->128) == [n,8192]x[8192,128], BatchNorm, L2Norm (HardNet.py:86-101, 12-19)
constexpr int HH_P = 16;  // patches per CTA
__global__ void __launch_bounds__(256) hardnet_head_kernel(const float* __restrict__ feat, const float* __restrict__ w,
                                                            const float* __restrict__ bn, float* __restrict__ out, int n,
                                                            int group, const int* __restrict__ count) {
    __shared__ float s_a[HH_P][64 + 1];
    const int p0 = blockIdx.x * HH_P;
    const int co = threadIdx.x & 127, half = threadIdx.x >> 7;  // half: patches [half*8, half*8+8)
    float acc[HH_P / 2];
#pragma unroll
    for (int k = 0; k < HH_P / 2; k++) acc[k] = 0.f;
    for (int k0 = 0; k0 < 8192; k0 += 64) {
        __syncthreads();
        for (int i = threadIdx.x; i < HH_P * 64; i += 256) {
            const int p = i >> 6, k = i & 63;
            s_a[p][k] = (p0 + p < n) ? feat[(size_t)(p0 + p) * 8192 + k0 + k] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 64; k++) {
            const float wv = __ldg(w + (size_t)(k0 + k) * 128 + co);
#pragma unroll
            for (int q = 0; q < HH_P / 2; q++) acc[q] = fmaf(s_a[half * (HH_P / 2) + q][k], wv, acc[q]);
        }
    }
    const float sc = bn[co], sh = bn[128 + co];
    float v[HH_P / 2];
#pragma unroll
    for (int q = 0; q < HH_P / 2; q++) v[q] = fmaf(acc[q], sc, sh);
    // sum of squares over the 128 channels of each patch: 4 warps per half, combined in a fixed order
    __syncthreads();
    const int wih = (threadIdx.x >> 5) & 3;  // warp index within the half
#pragma unroll
    for (int q = 0; q < HH_P / 2; q++) {
        const float ss = warp_sum(v[q] * v[q]);
        if ((threadIdx.x & 31) == 0) s_a[half * (HH_P / 2) + q][wih] = ss;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < HH_P / 2; q++) {
        const int r = half * (HH_P / 2) + q, p = p0 + r;
        if (p >= n) continue;
        if (count != nullptr && (p % group) >= count[p / group]) continue;
        const float ss = (s_a[r][0] + s_a[r][1]) + (s_a[r][2] + s_a[r][3]);
        out[(size_t)p * 128 + co] = v[q] / sqrtf(ss + 1e-8f);
    }
}

// ---- weight packing (host) ------------------------------------------------------------------------------
// Power of two that brings the largest |w| near 2^13.  The tensor-core engines store weights times this scale so that their
// fp16 residuals (w - fp16(w), 2^-11 of w) stay in fp16's normal range - below 6e-5 a residual would lose bits as a subnormal -
// and multiply the fp32 accumulators by the exact inverse.
static float pow2_scale(const float* w, size_t n) {
    float wmax = 0.f;
    for (size_t i = 0; i < n; i++) wmax = fmaxf(wmax, fabsf(w[i]));
    int ex = 0;
    if (wmax > 0.f) { frexpf(wmax, &ex); ex = 13 - ex; }
    return ldexpf(1.0f, ex);
}

static size_t blob_floats(int kind) {
    const LayerCfg* cfg = (kind == AG_NET_HARDNET) ? kHardCfg : kAffCfg;
    size_t n = 0;
    for (int l = 0; l < 6; l++) n += (size_t)cfg[l].cout * cfg[l].cin * 9 + 2 * cfg[l].cout;
    const int c = cfg[5].cout;
    if (kind == AG_NET_HARDNET) n += (size_t)128 * c * 64 + 256;
    else n += (size_t)(kind == AG_NET_AFFNET ? 3 : 2) * c * 64 + (kind == AG_NET_AFFNET ? 3 : 2);
    return n;
}

}  // namespace ag

using namespace ag;

extern "C" {

size_t ag_net_blob_floats(int kind) {
    if (kind < 0 || kind > 2) return 0;
    return blob_floats(kind);
}

int ag_net_create(int kind, const float* h_blob, size_t n_floats, ag_net_t** out) {
    AG_REQUIRE(out && h_blob, "NULL argument");
    AG_REQUIRE(kind >= 0 && kind <= 2, "unknown net kind");
    if (n_floats != blob_floats(kind)) {
        set_error("ag_net_create: blob has %zu floats, kind %d needs %zu", n_floats, kind, blob_floats(kind));
        return AG_ERR_INVALID;
    }
    const LayerCfg* cfg = (kind == AG_NET_HARDNET) ? kHardCfg : kAffCfg;
    std::vector<float> packed;
    size_t w_off[6], b_off[6], hw_off, hb_off;
    const float* p = h_blob;
    for (int l = 0; l < 6; l++) {
        const int ci = cfg[l].cin, co = cfg[l].cout;
        const float* w = p; const float* mean = w + (size_t)co * ci * 9; const float* var = mean + co;
        p = var + co;
        w_off[l] = packed.size();
        packed.resize(packed.size() + (size_t)9 * ci * co);
        float* dst = packed.data() + w_off[l];
        std::vector<float> invstd(co);
        for (int o = 0; o < co; o++) invstd[o] = 1.0f / sqrtf(var[o] + BN_EPS);
        for (int tap = 0; tap < 9; tap++)
            for (int c = 0; c < ci; c++)
                for (int o = 0; o < co; o++) dst[((size_t)tap * ci + c) * co + o] = w[((size_t)o * ci + c) * 9 + tap] * invstd[o];
        while (packed.size() % 4) packed.push_back(0.f);
        b_off[l] = packed.size();
        for (int o = 0; o < co; o++) packed.push_back(-mean[o] * invstd[o]);
        while (packed.size() % 4) packed.push_back(0.f);
    }
    const int c = cfg[5].cout;
    hw_off = packed.size();
    if (kind == AG_NET_HARDNET) {
        const float* w = p; const float* mean = w + (size_t)128 * c * 64; const float* var = mean + 128;
        packed.resize(packed.size() + (size_t)8192 * 128);
        float* dst = packed.data() + hw_off;
        for (int o = 0; o < 128; o++)
            for (int k = 0; k < 8192; k++) dst[(size_t)k * 128 + o] = w[(size_t)o * 8192 + k];
        hb_off = packed.size();
        for (int o = 0; o < 128; o++) packed.push_back(1.0f / sqrtf(var[o] + BN_EPS));
        for (int o = 0; o < 128; o++) packed.push_back(-mean[o] / sqrtf(var[o] + BN_EPS));
    } else {
        const int no = (kind == AG_NET_AFFNET) ? 3 : 2;
        const float* w = p; const float* bias = w + (size_t)no * c * 64;
        if (kind == AG_NET_ORINET) {
            // w_eff[k = ci*64 + y*8 + x][ch*9 + oy*3 + ox] = w[ch][ci][y-oy+1][x-ox+1] (zero outside the 8x8 kernel): padding = 1
            packed.resize(packed.size() + (size_t)4096 * 18);
            float* dst = packed.data() + hw_off;
            for (int ci = 0; ci < 64; ci++)
                for (int y = 0; y < 8; y++)
                    for (int x = 0; x < 8; x++)
                        for (int ch = 0; ch < 2; ch++)
                            for (int oy = 0; oy < 3; oy++)
                                for (int ox = 0; ox < 3; ox++) {
                                    const int ky = y - oy + 1, kx = x - ox + 1;
                                    const float v = (ky >= 0 && ky < 8 && kx >= 0 && kx < 8) ? w[((size_t)ch * 64 + ci) * 64 + ky * 8 + kx] : 0.f;
                                    dst[((size_t)ci * 64 + y * 8 + x) * 18 + ch * 9 + oy * 3 + ox] = v;
                                }
        } else
            packed.insert(packed.end(), w, w + (size_t)no * c * 64);
        hb_off = packed.size();
        packed.insert(packed.end(), bias, bias + no);
        while (packed.size() % 4) packed.push_back(0.f);
    }
    // power-of-two scales of the tensor-core weight packs, layers 1..6
    float w_scale[6];
    for (int l = 0; l < 6; l++) w_scale[l] = pow2_scale(packed.data() + w_off[l], (size_t)9 * cfg[l].cin * cfg[l].cout);
    // second-generation packs (tcx_pack_layer): kernel-row blocks with the three taps stacked along N
    std::vector<__half> packed_x;
    size_t wx_off[6] = {0, 0, 0, 0, 0, 0};
    for (int l = 1; l < 6; l++) {
        wx_off[l] = packed_x.size();
        tcx_pack_layer(packed.data() + w_off[l], cfg[l].cin, cfg[l].cout, tcx_stride(l), tcx_nsplit(kind, l), tcx_split_w(kind, l), w_scale[l], packed_x);
        while (packed_x.size() % 8) packed_x.push_back(__float2half_rn(0.f));
    }
    // HardNet: the same packs with bf16 operands (engine 5, BASELINE.json configs[4]) + the bf16 head weights
    std::vector<__half> packed_bf;
    size_t wbf_off[6] = {0, 0, 0, 0, 0, 0}, headbf_off = 0;
    if (kind == AG_NET_HARDNET) {
        for (int l = 1; l < 6; l++) {
            wbf_off[l] = packed_bf.size();
            tcx_pack_layer(packed.data() + w_off[l], cfg[l].cin, cfg[l].cout, tcx_stride(l), tcx_nsplit(kind, l), tcx_split_w(kind, l), w_scale[l], packed_bf, 1);
            while (packed_bf.size() % 8) packed_bf.push_back(__float2half_rn(0.f));
        }
        headbf_off = packed_bf.size();
        packed_bf.resize(packed_bf.size() + (size_t)8192 * 128);
        const float* hw = packed.data() + hw_off;  // [k = c*64 + p][cout]
        for (int pix = 0; pix < 64; pix++)
            for (int cg = 0; cg < 16; cg++)
                for (int o = 0; o < 128; o++)
                    for (int e = 0; e < 8; e++) {
                        const __nv_bfloat16 bv = __float2bfloat16_rn(hw[((size_t)(cg * 8 + e) * 64 + pix) * 128 + o]);
                        memcpy(&packed_bf[headbf_off + (((size_t)(pix * 16 + cg)) * 128 + o) * 8 + e], &bv, 2);
                    }
    }
    // fp16 head packs for the tensor-core head GEMMs
    std::vector<__half> packed_h;
    float head_scale = 1.0f;
    if (kind == AG_NET_HARDNET) {
        packed_h.resize((size_t)8192 * 128);
        __half* dst = packed_h.data();
        const float* hw = packed.data() + hw_off;  // [k = c*64 + p][cout]
        for (int pix = 0; pix < 64; pix++)
            for (int cg = 0; cg < 16; cg++)
                for (int o = 0; o < 128; o++)
                    for (int e = 0; e < 8; e++)
                        dst[(((size_t)(pix * 16 + cg)) * 128 + o) * 8 + e] = __float2half_rn(hw[((size_t)(cg * 8 + e) * 64 + pix) * 128 + o]);
    }
    if (kind != AG_NET_HARDNET) {   // AffNet (3 outputs) / OriNet (18 shifted outputs): [4096/8][32 hi rows | 32 lo rows][8]
        const int no = (kind == AG_NET_AFFNET) ? 3 : 18;
        packed_h.resize((size_t)4096 * 64, __float2half_rn(0.f));
        __half* dst = packed_h.data();
        const float* hw = packed.data() + hw_off;
        // the weights are stored times a power of two that brings the largest one near 2^13: their fp16 residuals then stay in
        // the normal range (a residual below 6e-5 would lose bits as a subnormal); the epilogue multiplies by 1/scale, exactly
        head_scale = pow2_scale(hw, (size_t)4096 * no);
        for (int pix = 0; pix < 64; pix++)
            for (int cg = 0; cg < 8; cg++)
                for (int o = 0; o < no; o++)
                    for (int e = 0; e < 8; e++) {
                        const size_t k = (size_t)(cg * 8 + e) * 64 + pix;
                        const float v = head_scale * ((kind == AG_NET_AFFNET) ? hw[(size_t)o * 4096 + k] : hw[k * 18 + o]);
                        const __half hi = __float2half_rn(v);
                        const size_t chunk = (size_t)pix * 8 + cg;
                        dst[(chunk * 64 + o) * 8 + e] = hi;
                        dst[(chunk * 64 + 32 + o) * 8 + e] = __float2half_rn(v - __half2float(hi));
                    }
    }
    ag_net* net = new ag_net();
    memset(net, 0, sizeof(*net));
    net->kind = kind;
    net->engine = AG_ENGINE_TC2;   // tensor-core engine (nets_tcx.cu)
    net->head_inv_scale = 1.0f / head_scale;
    for (int l = 0; l < 6; l++) net->w_inv_scale[l] = 1.0f / w_scale[l];
    {
        int rch = check_cuda(cudaMalloc(&net->d_all_h, packed_h.size() * sizeof(__half)), "cudaMalloc fp16 weights");
        if (rch != AG_OK) { delete net; return rch; }
        rch = check_cuda(cudaMemcpy(net->d_all_h, packed_h.data(), packed_h.size() * sizeof(__half), cudaMemcpyHostToDevice), "upload fp16 weights");
        if (rch != AG_OK) { cudaFree(net->d_all_h); delete net; return rch; }
        net->d_headh = net->d_all_h;
        rch = check_cuda(cudaMalloc(&net->d_all_x, packed_x.size() * sizeof(__half)), "cudaMalloc fp16 weights (second generation)");
        if (rch == AG_OK) rch = check_cuda(cudaMemcpy(net->d_all_x, packed_x.data(), packed_x.size() * sizeof(__half), cudaMemcpyHostToDevice), "upload fp16 weights");
        if (rch != AG_OK) { cudaFree(net->d_all_h); cudaFree(net->d_all_x); delete net; return rch; }
        for (int l = 1; l < 6; l++) net->d_wx[l] = net->d_all_x + wx_off[l];
        if (!packed_bf.empty()) {   // appended behind the fp16 packs in a second allocation owned through d_wx_bf[0]
            __half* dbf = nullptr;
            rch = check_cuda(cudaMalloc(&dbf, packed_bf.size() * sizeof(__half)), "cudaMalloc bf16 weights");
            if (rch == AG_OK) rch = check_cuda(cudaMemcpy(dbf, packed_bf.data(), packed_bf.size() * sizeof(__half), cudaMemcpyHostToDevice), "upload bf16 weights");
            if (rch != AG_OK) { cudaFree(dbf); cudaFree(net->d_all_h); cudaFree(net->d_all_x); delete net; return rch; }
            net->d_wx_bf[0] = dbf;
            for (int l = 1; l < 6; l++) net->d_wx_bf[l] = dbf + wbf_off[l];
            net->d_headh_bf = dbf + headbf_off;
        }
    }
    int rc = check_cuda(cudaMalloc(&net->d_all, packed.size() * sizeof(float)), "cudaMalloc weights");
    if (rc != AG_OK) { cudaFree(net->d_all_h); cudaFree(net->d_all_x); delete net; return rc; }
    rc = check_cuda(cudaMemcpy(net->d_all, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice), "upload weights");
    if (rc != AG_OK) { cudaFree(net->d_all); cudaFree(net->d_all_h); cudaFree(net->d_all_x); delete net; return rc; }
    for (int l = 0; l < 6; l++) { net->d_w[l] = net->d_all + w_off[l]; net->d_b[l] = net->d_all + b_off[l]; }
    net->d_w1 = net->d_w[0];
    net->d_head_w = net->d_all + hw_off;
    net->d_head_b = net->d_all + hb_off;
    *out = net;
    return AG_OK;
}

void ag_net_destroy(ag_net_t* net) {
    if (!net) return;
    cudaFree(net->d_all);
    cudaFree(net->d_all_h);
    cudaFree(net->d_all_x);
    cudaFree(net->d_wx_bf[0]);
    delete net;
}

int ag_net_set_engine(ag_net_t* net, int engine) {
    AG_REQUIRE(net != nullptr, "NULL net");
    AG_REQUIRE(engine == AG_ENGINE_SIMT || engine == AG_ENGINE_TC2 || engine == AG_ENGINE_TC2_BF16, "unknown engine");
    AG_REQUIRE(engine != AG_ENGINE_TC2_BF16 || net->kind == AG_NET_HARDNET, "the bf16 engine exists for HardNet only");
    net->engine = engine;
    return AG_OK;
}

int ag_net_get_engine(const ag_net_t* net) { return net ? net->engine : -1; }

size_t ag_net_workspace_bytes(int kind, int n) {
    if (n <= 0) return 0;
    const size_t per = (kind == AG_NET_HARDNET) ? 32768 : 16384;  // largest fp32 activation per patch (floats), SIMT engine
    const size_t simt = 2 * align_up((size_t)n * per * sizeof(float), 256);
    // tensor-core engine: two fp16 ping-pong buffers + the hi/lo fp16 head operand (AffNet/OriNet, whole 128-patch tiles) or the fp16 head operand (HardNet, padded
    // to a multiple of 128 patches)
    const size_t tcb = 2 * align_up(tcx_act_bytes(n), 256) +
                       (kind == AG_NET_HARDNET ? align_up(((size_t)n + 128) * 8192 * 2, 256) : align_up(tc_headx_bytes(n), 256));
    return simt > tcb ? simt : tcb;
}

}  // extern "C"

namespace ag {

static int trunk_affnet(const ag_net* net, const float* patches, int n, int group, const int* count, float* a, float* b,
                        cudaStream_t st) {
    int rc;
    if ((rc = launch_conv<1, 16, 32, 1, 16, 1, true>(patches, a, net->d_w[0], net->d_b[0], n, group, count, st))) return rc;
    if ((rc = launch_conv<16, 16, 32, 1, 16, 16, false>(a, b, net->d_w[1], net->d_b[1], n, group, count, st))) return rc;
    if ((rc = launch_conv<16, 32, 32, 2, 32, 16, false>(b, a, net->d_w[2], net->d_b[2], n, group, count, st))) return rc;
    if ((rc = launch_conv<32, 32, 16, 1, 32, 32, false>(a, b, net->d_w[3], net->d_b[3], n, group, count, st))) return rc;
    if ((rc = launch_conv<32, 64, 16, 2, 64, 32, false>(b, a, net->d_w[4], net->d_b[4], n, group, count, st))) return rc;
    if ((rc = launch_conv<64, 64, 8, 1, 64, 32, false>(a, b, net->d_w[5], net->d_b[5], n, group, count, st))) return rc;
    return AG_OK;  // features in b: [n,64,8,8]
}

static int trunk_hardnet(const ag_net* net, const float* patches, int n, int group, const int* count, float* a, float* b,
                         cudaStream_t st) {
    int rc;
    if ((rc = launch_conv<1, 32, 32, 1, 32, 1, true>(patches, a, net->d_w[0], net->d_b[0], n, group, count, st))) return rc;
    if ((rc = launch_conv<32, 32, 32, 1, 32, 32, false>(a, b, net->d_w[1], net->d_b[1], n, group, count, st))) return rc;
    if ((rc = launch_conv<32, 64, 32, 2, 64, 32, false>(b, a, net->d_w[2], net->d_b[2], n, group, count, st))) return rc;
    if ((rc = launch_conv<64, 64, 16, 1, 64, 32, false>(a, b, net->d_w[3], net->d_b[3], n, group, count, st))) return rc;
    if ((rc = launch_conv<64, 128, 16, 2, 128, 16, false>(b, a, net->d_w[4], net->d_b[4], n, group, count, st))) return rc;
    if ((rc = launch_conv<128, 128, 8, 1, 128, 16, false>(a, b, net->d_w[5], net->d_b[5], n, group, count, st))) return rc;
    return AG_OK;  // features in b: [n,128,8,8]
}

// Runs the six conv layers with the net's engine; *feat receives the feature pointer: fp32 NCHW [n,C,8,8] (SIMT engine) or the
// fp16 hi/lo head-GEMM operand (tensor-core engines).
static int run_trunk(const ag_net* net, const float* patches, const tc::FirstSrc* pyr_src, int n, int group, const int* count, float* a,
                     float* b, float** feat, cudaStream_t st) {
    if (net->engine != AG_ENGINE_SIMT) {
        const tc::FirstSrc src = pyr_src ? *pyr_src : tc_src_patches(patches);
        // the workspace [a, a + 2*(b-a)) is re-carved as [bufA | bufB | head-GEMM operand]
        char* base = (char*)a;
        const size_t total = 2 * (size_t)((char*)b - (char*)a);
        const size_t act = align_up(tcx_act_bytes(n), 256);
        const size_t fbytes = tc_headx_bytes(n);
        if (2 * act + fbytes > total) { set_error("tensor-core workspace too small"); return AG_ERR_CAPACITY; }
        void* bufA = base;
        void* bufB = base + act;
        b = (float*)(base + 2 * act);
        *feat = b;
        if (net->kind == AG_NET_HARDNET) { set_error("HardNet tensor-core path has its own entry"); return AG_ERR_INVALID; }
        return tcx_trunk_affori(net, src, n, group, count, bufA, bufB, b, st, 6);
    }
    *feat = b;
    if (patches == nullptr) { set_error("the fp32 SIMT engine needs materialised patches"); return AG_ERR_INVALID; }
    return net->kind == AG_NET_HARDNET ? trunk_hardnet(net, patches, n, group, count, a, b, st)
                                       : trunk_affnet(net, patches, n, group, count, a, b, st);
}

static int split_ws(int kind, int n, void* d_ws, size_t ws_bytes, float** a, float** b) {
    const size_t need = ag_net_workspace_bytes(kind, n);
    if (d_ws == nullptr || ws_bytes < need) {
        set_error("net forward: workspace of %zu bytes needed, %zu given", need, ws_bytes);
        return AG_ERR_CAPACITY;
    }
    *a = (float*)d_ws;
    *b = (float*)((char*)d_ws + need / 2);
    return AG_OK;
}

}  // namespace ag

extern "C" {

static int affnet_impl(const ag_net_t* net, const float* d_patches, const tc::FirstSrc* src, int n, const int* d_count, int group,
                       float* d_out, void* d_ws, size_t ws_bytes, void* stream, float* d_raw = nullptr) {
    AG_REQUIRE(net && (d_patches || src) && (d_out || d_raw), "NULL argument");
    AG_REQUIRE(net->kind == AG_NET_AFFNET, "not an AffNet handle");
    if (n <= 0) return AG_OK;
    if (group <= 0) group = n;
    float *a, *b;
    int rc = split_ws(net->kind, n, d_ws, ws_bytes, &a, &b);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = run_trunk(net, d_patches, src, n, group, d_count, a, b, &b, st))) return rc;
    if (net->engine == AG_ENGINE_TC2) return tc_headx_forward(net, b, n, group, d_count, d_out, nullptr, st, d_raw);
    AG_REQUIRE(d_raw == nullptr && d_out, "raw head outputs need the tensor-core engine (4)");
    affnet_head_kernel<<<cdiv(n, 8), 256, 0, st>>>(b, net->d_head_w, net->d_head_b, d_out, n, group, d_count);
    AG_CHECK_LAUNCH("affnet_head_kernel");
    return AG_OK;
}

static int orinet_impl(const ag_net_t* net, const float* d_patches, const tc::FirstSrc* src, int n, const int* d_count, int group,
                       float* d_out, float* d_angle, void* d_ws, size_t ws_bytes, void* stream, float* d_raw = nullptr) {
    AG_REQUIRE(net && (d_patches || src) && (d_out || d_angle || d_raw), "NULL argument");
    AG_REQUIRE(net->kind == AG_NET_ORINET, "not an OriNet handle");
    if (n <= 0) return AG_OK;
    if (group <= 0) group = n;
    float *a, *b;
    int rc = split_ws(net->kind, n, d_ws, ws_bytes, &a, &b);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = run_trunk(net, d_patches, src, n, group, d_count, a, b, &b, st))) return rc;
    if (net->engine == AG_ENGINE_TC2) return tc_headx_forward(net, b, n, group, d_count, d_out, d_angle, st, d_raw);
    AG_REQUIRE(d_raw == nullptr, "raw head outputs need the tensor-core engine (4)");
    orinet_head_kernel<<<cdiv(n, OH_W * OH_P), OH_W * 32, 0, st>>>(b, net->d_head_w, net->d_head_b, d_out, d_angle, n, group, d_count);
    AG_CHECK_LAUNCH("orinet_head_kernel");
    return AG_OK;
}

static int hardnet_impl(const ag_net_t* net, const float* d_patches, const tc::FirstSrc* src, int n, const int* d_count, int group,
                        float* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(net && (d_patches || src) && d_out, "NULL argument");
    AG_REQUIRE(net->kind == AG_NET_HARDNET, "not a HardNet handle");
    if (n <= 0) return AG_OK;
    if (group <= 0) group = n;
    float *a, *b;
    int rc = split_ws(net->kind, n, d_ws, ws_bytes, &a, &b);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (net->engine == AG_ENGINE_TC2 || net->engine == AG_ENGINE_TC2_BF16) {
        const int bf = net->engine == AG_ENGINE_TC2_BF16;
        char* base = (char*)d_ws;
        const size_t act = align_up(tcx_act_bytes(n), 256);
        const tc::FirstSrc s0 = src ? *src : tc_src_patches(d_patches);
        if ((rc = tcx_trunk_hardnet(net, s0, n, group, d_count, base, base + act, base + 2 * act, st, 6, bf))) return rc;
        return tc_hardnet_head(net, base + 2 * act, n, group, d_count, d_out, st, bf);
    }
    if ((rc = run_trunk(net, d_patches, src, n, group, d_count, a, b, &b, st))) return rc;
    hardnet_head_kernel<<<cdiv(n, HH_P), 256, 0, st>>>(b, net->d_head_w, net->d_head_b, d_out, n, group, d_count);
    AG_CHECK_LAUNCH("hardnet_head_kernel");
    return AG_OK;
}

int ag_affnet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out, void* d_ws,
                      size_t ws_bytes, void* stream) {
    AG_REQUIRE(d_patches, "NULL patches");
    return affnet_impl(net, d_patches, nullptr, n, d_count, group, d_out, d_ws, ws_bytes, stream);
}
int ag_orinet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out, float* d_angle,
                      void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(d_patches, "NULL patches");
    return orinet_impl(net, d_patches, nullptr, n, d_count, group, d_out, d_angle, d_ws, ws_bytes, stream);
}
/* Raw head outputs, the TorchScript modules' contract (convertJIT/AffNetJIT.pt: xy + [1, 0, 1] -> [n,3]; OriNetJIT.pt: xy -> [n,2]). */
int ag_affnet_forward_raw(const ag_net_t* net, const float* d_patches, int n, float* d_raw, void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(d_patches && d_raw, "NULL argument");
    return affnet_impl(net, d_patches, nullptr, n, nullptr, n, nullptr, d_ws, ws_bytes, stream, d_raw);
}
int ag_orinet_forward_raw(const ag_net_t* net, const float* d_patches, int n, float* d_raw, void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(d_patches && d_raw, "NULL argument");
    return orinet_impl(net, d_patches, nullptr, n, nullptr, n, nullptr, nullptr, d_ws, ws_bytes, stream, d_raw);
}
int ag_hardnet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out, void* d_ws,
                       size_t ws_bytes, void* stream) {
    AG_REQUIRE(d_patches, "NULL patches");
    return hardnet_impl(net, d_patches, nullptr, n, d_count, group, d_out, d_ws, ws_bytes, stream);
}

// Fused sampler + net: patches are sampled from the pyramid inside the first tensor-core layer (tensor-core engine only).
int ag_net_forward_pyr(const ag_net_t* net, const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                       const int* d_lvl, const int* d_count, int cap, float* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    AG_REQUIRE(net && plan && d_pyr && d_lafs && d_oct && d_lvl && d_out, "NULL argument");
    AG_REQUIRE(cap >= 1, "bad capacity");
    AG_REQUIRE(net->engine != AG_ENGINE_SIMT, "fused sampling needs a tensor-core engine");
    const tc::FirstSrc src = tc_src_pyramid(plan, d_pyr, d_lafs, d_oct, d_lvl, cap);
    const int n = plan->B * cap;
    if (net->kind == AG_NET_AFFNET) return affnet_impl(net, nullptr, &src, n, d_count, cap, d_out, d_ws, ws_bytes, stream);
    if (net->kind == AG_NET_ORINET) return orinet_impl(net, nullptr, &src, n, d_count, cap, d_out, nullptr, d_ws, ws_bytes, stream);
    return hardnet_impl(net, nullptr, &src, n, d_count, cap, d_out, d_ws, ws_bytes, stream);
}

}  // extern "C"
