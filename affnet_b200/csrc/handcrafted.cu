// Hand-crafted orientation and affine shape (SURVEY.md §8(f) rows 1 and 2): the estimators the reference uses when no OriNet /
// AffNet is given.  Replaces OrientationDetector.forward (HandCraftedModules.py:168-192) and AffineShapeEstimator.forward
// (HandCraftedModules.py:94-132).  One warp per patch; the patch (PS x PS, PS <= 41) is staged in shared memory.
#include <math.h>

#include "common.cuh"

namespace ag {

constexpr int HC_MAXPS = 41, HC_WARPS = 2, HCP_WARPS = 4;   // HCP: the pyramid-sampling kernels

__device__ __forceinline__ float warp_sum_f(float v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// gradient with replicate padding; wx = (w_minus, w_plus) of the (1x3) cross-correlation
__device__ __forceinline__ void grad_at(const float* p, int PS, int i, int j, float wm, float wp, float& gx, float& gy) {
    const int jm = max(j - 1, 0), jp = min(j + 1, PS - 1), im = max(i - 1, 0), ip = min(i + 1, PS - 1);
    gx = __fadd_rn(__fmul_rn(wm, p[i * PS + jm]), __fmul_rn(wp, p[i * PS + jp]));
    gy = __fadd_rn(__fmul_rn(wm, p[im * PS + j]), __fmul_rn(wp, p[ip * PS + j]));
}

// OrientationDetector.forward (HandCraftedModules.py:168-192) on a PS x PS patch p in shared memory: per-pixel lower bin and weight
// (s_b, s_w [NP]), per-bin sums in raster order, / NP, (0.33, 0.34, 0.33) smoothing (s_h [40]), first maximum -> angle, on every lane.
// Shared by orientation_hist_kernel and orientation_hist_pyr_kernel, so both give the same bits.
__device__ __forceinline__ float orientation_of_patch(const float* p, int PS, const float* gk, unsigned char* s_b, float* s_w, float* s_h,
                                                      int lane) {
    const int NP = PS * PS;
    const float PI_F = 3.14159265358979323846f;
    for (int i = lane; i < NP; i += 32) {
        float gx, gy;
        grad_at(p, PS, i / PS, i % PS, 0.5f, -0.5f, gx, gy);   // weights (0.5, 0, -0.5): 0.5*x[j-1] - 0.5*x[j+1]
        const float mag = __fmul_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), 1e-10f)), gk[i]);
        const float ori = atan2f(gy, gx);
        const float o_big = __fdiv_rn(__fmul_rn(36.0f, __fadd_rn(ori, PI_F)), 2.0f * PI_F);
        float bo0 = floorf(o_big);
        const float wo1 = __fsub_rn(o_big, bo0);
        bo0 = fmodf(bo0, 36.0f);
        s_b[i] = (unsigned char)(int)bo0;
        s_w[i] = __fmul_rn(__fsub_rn(1.0f, wo1), mag);   // only the lower-bin weight is accumulated (as the reference does)
    }
    __syncwarp();
    // deterministic histogram: lane b sums bin b (and b+32) over all pixels in raster order
    for (int b = lane; b < 36; b += 32) {
        float acc = 0.f;
        for (int i = 0; i < NP; i++)
            if (s_b[i] == b) acc += s_w[i];
        s_h[b + 1] = acc / (float)NP;   // adaptive_avg_pool2d -> mean
    }
    if (lane == 0) { s_h[0] = 0.f; s_h[37] = 0.f; }   // conv1d zero padding
    __syncwarp();
    float best = -INFINITY;
    int bidx = 0;
    for (int b = lane; b < 36; b += 32) {
        const float v = fmaf(0.33f, s_h[b + 2], fmaf(0.34f, s_h[b + 1], 0.33f * s_h[b]));
        if (v > best) { best = v; bidx = b; }
    }
    // first maximum wins (torch.max on CPU)
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
    }
    return -__fsub_rn(__fdiv_rn(__fmul_rn(2.0f * PI_F, (float)bidx), 36.0f), PI_F);
}

// AffineShapeEstimator.forward (HandCraftedModules.py:94-132) on a PS x PS patch p in shared memory: Gaussian-weighted second moments
// (lane-strided pixel walk, butterfly sum), invSqrt, abc2A + up-is-up rectification -> A, on every lane.  Shared by baumberg_kernel
// and baumberg_pyr_kernel, so both give the same bits.
__device__ __forceinline__ void baumberg_of_patch(const float* p, int PS, const float* gk, int lane, float (&A)[4]) {
    const int NP = PS * PS;
    float a = 0.f, b = 0.f, c = 0.f;
    for (int i = lane; i < NP; i += 32) {
        float gx, gy;
        grad_at(p, PS, i / PS, i % PS, -1.0f, 1.0f, gx, gy);   // weights (-1, 0, 1)
        const float g = gk[i];
        a += gx * gx * g; b += gx * gy * g; c += gy * gy * g;
    }
    a = warp_sum_f(a) / (float)NP; b = warp_sum_f(b) / (float)NP; c = warp_sum_f(c) / (float)NP;
    // invSqrt (HandCraftedModules.py:94-117)
    const float eps = 1e-12f;
    const float mask = (b != 0.f) ? 1.f : 0.f;
    const float r1 = mask * (c - a) / (2.f * b + eps);
    const float sgn = (r1 > 0.f) ? 1.f : ((r1 < 0.f) ? -1.f : 0.f);
    const float t1 = sgn / (fabsf(r1) + sqrtf(1.f + r1 * r1));
    float r = 1.0f / sqrtf(1.f + t1 * t1);
    float t = t1 * r;
    r = r * mask + 1.0f * (1.0f - mask);
    t = t * mask;
    float x = 1.f / sqrtf(r * r * a - 2.0f * r * t * b + t * t * c);
    float z = 1.f / sqrtf(t * t * a + 2.0f * r * t * b + r * r * c);
    const float d = sqrtf(x * z);
    x = x / d; z = z / d;
    const float na = r * r * x + t * t * z, nb = -r * t * x + t * r * z, nc = t * t * x + r * r * z;
    // abc2A + rectifyAffineTransformationUpIsUp (LAF.py:285-291)
    const float a00 = na, a01 = nb, a10 = nb, a11 = nc;
    const float det = sqrtf(fabsf(a00 * a11 - a10 * a01 + 1e-10f));
    const float b2a2 = sqrtf(a01 * a01 + a00 * a00);
    A[0] = b2a2 / det; A[1] = 0.f;
    A[2] = (a11 * a01 + a10 * a00) / (b2a2 * det); A[3] = det / b2a2;
}

__global__ void __launch_bounds__(HC_WARPS * 32) orientation_hist_kernel(const float* __restrict__ patches, int n, int PS, const float* __restrict__ gk,
                                                                        float* __restrict__ angle) {
    __shared__ float s_p[HC_WARPS][HC_MAXPS * HC_MAXPS];
    __shared__ float s_w[HC_WARPS][HC_MAXPS * HC_MAXPS];
    __shared__ unsigned char s_b[HC_WARPS][HC_MAXPS * HC_MAXPS];
    __shared__ float s_h[HC_WARPS][40];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pi = blockIdx.x * HC_WARPS + warp;
    if (pi >= n) return;
    const int NP = PS * PS;
    float* p = s_p[warp];
    for (int i = lane; i < NP; i += 32) p[i] = patches[(size_t)pi * NP + i];
    __syncwarp();
    const float ang = orientation_of_patch(p, PS, gk, s_b[warp], s_w[warp], s_h[warp], lane);
    if (lane == 0) angle[pi] = ang;
}

__global__ void __launch_bounds__(HC_WARPS * 32) baumberg_kernel(const float* __restrict__ patches, int n, int PS, const float* __restrict__ gk,
                                                                float* __restrict__ A) {
    __shared__ float s_p[HC_WARPS][HC_MAXPS * HC_MAXPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pi = blockIdx.x * HC_WARPS + warp;
    if (pi >= n) return;
    const int NP = PS * PS;
    float* p = s_p[warp];
    for (int i = lane; i < NP; i += 32) p[i] = patches[(size_t)pi * NP + i];
    __syncwarp();
    float a[4];
    baumberg_of_patch(p, PS, gk, lane, a);
    if (lane != 0) return;
    float* o = A + (size_t)pi * 4;
    o[0] = a[0]; o[1] = a[1]; o[2] = a[2]; o[3] = a[3];
}

// ---- the same estimators sampling their patches from the pyramid (the batched pipeline's path) --------------------------------------
// Row r = b * cap + i is LAF i of image b, sampled at pyr[oct[r]][lvl[r]] exactly as extract_patches_pyr_kernel does; rows i >= count[b]
// are skipped.  One warp per keypoint; the PS x PS patch lives only in shared memory.  The Gaussian window (fully determined by PS)
// comes in the parameter struct and is staged once per block.
struct HcPyrArgs {
    PyrGeom G;
    float gk[HC_MAXPS * HC_MAXPS];
};

// Shared-memory layout: window [NP] floats, then per warp the patch [NP] (+ orientation: weights [NP], histogram [40]), then per warp the
// orientation's bin bytes [NP].
__host__ __device__ inline int hcp_warp_floats(int PS, bool ori) { return PS * PS * (ori ? 2 : 1) + (ori ? 40 : 0); }
inline size_t hcp_smem_bytes(int PS, bool ori) {
    return sizeof(float) * (size_t)(PS * PS + HCP_WARPS * hcp_warp_floats(PS, ori)) + (ori ? (size_t)HCP_WARPS * PS * PS : 0);
}

// Samples the PS x PS patch of the normalised LAF Lr at level (o, l) of image b into p (lane-strided), as extract_patches_pyr_kernel does.
__device__ __forceinline__ void sample_row_patch(const PyrGeom& G, const float* __restrict__ pyr, const float (&Lr)[6], int o, int l, int b,
                                                 int PS, int lane, float* p) {
    const int h = G.h[o], w = G.w[o];
    const float* img = pyr + G.off[o][l] + (size_t)b * h * w;
    const int NP = PS * PS;
    for (int t = lane; t < NP; t += 32) {
        const int i = t / PS, j = t - i * PS;
        float px, py;
        laf_sample_xy(Lr, h, w, i, j, 1.0f / (float)PS, px, py);
        p[t] = bilinear_zero(img, h, w, px, py);
    }
}

__global__ void __launch_bounds__(HCP_WARPS * 32) orientation_hist_pyr_kernel(const HcPyrArgs P, const float* __restrict__ pyr, const float* lafs,
                                                                             const int* __restrict__ oct, const int* __restrict__ lvl,
                                                                             const int* __restrict__ count, int cap, int PS,
                                                                             float* __restrict__ angle, float* lafs_out) {
    extern __shared__ float hc_smem[];
    const int NP = PS * PS;
    float* s_gk = hc_smem;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) s_gk[i] = P.gk[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * HCP_WARPS + warp;
    if (row >= P.G.B * cap) return;
    const int b = row / cap;
    if (count != nullptr && row - b * cap >= count[b]) return;
    float* p = hc_smem + NP + warp * hcp_warp_floats(PS, true);
    float* s_w = p + NP;
    float* s_h = s_w + NP;
    unsigned char* s_b = (unsigned char*)(hc_smem + NP + HCP_WARPS * hcp_warp_floats(PS, true)) + warp * NP;
    float Lr[6];
#pragma unroll
    for (int q = 0; q < 6; q++) Lr[q] = lafs[(size_t)row * 6 + q];
    const int o = clampi(oct[row], 0, P.G.n_octaves - 1), l = clampi(lvl[row], 0, P.G.n_levels - 1);
    sample_row_patch(P.G, pyr, Lr, o, l, b, PS, lane, p);
    __syncwarp();
    const float ang = orientation_of_patch(p, PS, s_gk, s_b, s_w, s_h, lane);
    if (lane != 0) return;
    if (angle) angle[row] = ang;
    if (lafs_out) {   // angles2A (LAF.py:306-311): R = [[cos, sin], [-sin, cos]], then LAF_A <- LAF_A R
        const float c = cosf(ang), s = sinf(ang);
        laf_rotate(Lr, c, s, -s, c);
#pragma unroll
        for (int q = 0; q < 6; q++) lafs_out[(size_t)row * 6 + q] = Lr[q];
    }
}

// All n_iters Baumberg iterations of getAffineShape (SparseImgRepresenter.py:155-166) in one launch: sample at the working LAF, one
// Baumberg step, base_A <- A base_A, working LAF <- [base_A LAF_A | t].  base_A and the working LAF stay in registers.
__global__ void __launch_bounds__(HCP_WARPS * 32) baumberg_pyr_kernel(const HcPyrArgs P, const float* __restrict__ pyr, const float* __restrict__ lafs,
                                                                     const int* __restrict__ oct, const int* __restrict__ lvl,
                                                                     const int* __restrict__ count, int cap, int PS, int n_iters,
                                                                     float* __restrict__ A_out) {
    extern __shared__ float hc_smem[];
    const int NP = PS * PS;
    float* s_gk = hc_smem;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) s_gk[i] = P.gk[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * HCP_WARPS + warp;
    if (row >= P.G.B * cap) return;
    const int b = row / cap;
    if (count != nullptr && row - b * cap >= count[b]) return;
    float* p = hc_smem + NP + warp * hcp_warp_floats(PS, false);
    float L0[6], cur[6];
#pragma unroll
    for (int q = 0; q < 6; q++) cur[q] = L0[q] = lafs[(size_t)row * 6 + q];
    const int o = clampi(oct[row], 0, P.G.n_octaves - 1), l = clampi(lvl[row], 0, P.G.n_levels - 1);
    float base[4];
    for (int it = 0; it < n_iters; it++) {
        sample_row_patch(P.G, pyr, cur, o, l, b, PS, lane, p);
        __syncwarp();
        float A[4];
        baumberg_of_patch(p, PS, s_gk, lane, A);
        if (it == 0) {
#pragma unroll
            for (int q = 0; q < 4; q++) base[q] = A[q];
        } else {
            float nb[4];
            mat2_mul(A, base, nb);
#pragma unroll
            for (int q = 0; q < 4; q++) base[q] = nb[q];
        }
        if (it != n_iters - 1) laf_left_mul(base, L0, cur);
        __syncwarp();   // every lane is done with p before the next sample overwrites it
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 4; q++) A_out[(size_t)row * 4 + q] = base[q];
    }
}

}  // namespace ag

using namespace ag;

extern "C" {

int ag_circular_gauss_kernel(int kernlen, double sigma, float* h_out) {
    AG_REQUIRE(h_out && kernlen >= 1, "bad arguments");
    // CircularGaussKernel(kernlen, sigma, circ_zeros=False, norm=True) under python3 (Utils.py:92-114)
    const double half = kernlen / 2.0, r2 = half * half;
    const double sigma2 = (sigma > 0.0) ? 2.0 * sigma * sigma : 0.9 * r2;
    const double step = (kernlen > 1) ? (2.0 * half) / (kernlen - 1) : 0.0;
    double sum = 0.0;
    for (int i = 0; i < kernlen; i++)
        for (int j = 0; j < kernlen; j++) {
            const double y = (i == kernlen - 1) ? half : -half + i * step, x = (j == kernlen - 1) ? half : -half + j * step;
            sum += exp(-(x * x + y * y) / sigma2);
        }
    for (int i = 0; i < kernlen; i++)
        for (int j = 0; j < kernlen; j++) {
            const double y = (i == kernlen - 1) ? half : -half + i * step, x = (j == kernlen - 1) ? half : -half + j * step;
            h_out[i * kernlen + j] = (float)(exp(-(x * x + y * y) / sigma2) / sum);
        }
    return AG_OK;
}

int ag_orientation_hist(const float* d_patches, int n, int PS, const float* d_gk, float* d_angle, void* stream) {
    AG_REQUIRE(d_patches && d_gk && d_angle, "NULL argument");
    AG_REQUIRE(PS >= 3 && PS <= HC_MAXPS, "patch size out of range (3..41)");
    if (n <= 0) return AG_OK;
    orientation_hist_kernel<<<cdiv(n, HC_WARPS), HC_WARPS * 32, 0, (cudaStream_t)stream>>>(d_patches, n, PS, d_gk, d_angle);
    AG_CHECK_LAUNCH("orientation_hist_kernel");
    return AG_OK;
}

int ag_baumberg_shape(const float* d_patches, int n, int PS, const float* d_gk, float* d_A, void* stream) {
    AG_REQUIRE(d_patches && d_gk && d_A, "NULL argument");
    AG_REQUIRE(PS >= 3 && PS <= HC_MAXPS, "patch size out of range (3..41)");
    if (n <= 0) return AG_OK;
    baumberg_kernel<<<cdiv(n, HC_WARPS), HC_WARPS * 32, 0, (cudaStream_t)stream>>>(d_patches, n, PS, d_gk, d_A);
    AG_CHECK_LAUNCH("baumberg_kernel");
    return AG_OK;
}

// The windows are computed here, on the host, exactly as the modules compute theirs (HandCraftedModules.py _gauss_window: float32
// CircularGaussKernel times the scale), and travel in the kernel parameters: no device allocation or copy, so the launch is capturable.
static void hcp_args(const ag_pyramid_plan_t* plan, int PS, double sigma, float scale, HcPyrArgs& P) {
    P.G = make_geom(plan);
    ag_circular_gauss_kernel(PS, sigma, P.gk);
    for (int i = 0; i < PS * PS; i++) P.gk[i] = P.gk[i] * scale;
}

int ag_orientation_hist_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct, const int* d_lvl,
                            const int* d_count, int cap, int PS, float* d_angle, float* d_lafs_out, void* stream) {
    AG_REQUIRE(plan && d_pyr && d_lafs && d_oct && d_lvl && (d_angle || d_lafs_out), "NULL argument");
    AG_REQUIRE(PS >= 3 && PS <= HC_MAXPS, "patch size out of range (3..41)");
    AG_REQUIRE(cap >= 1 && (long long)plan->B * cap <= (1ll << 30), "bad sizes");
    HcPyrArgs P;
    hcp_args(plan, PS, 0.0, 10.0f, P);   // OrientationDetector: 10 x CircularGaussKernel(PS)
    const size_t smem = hcp_smem_bytes(PS, true);
    static SmemAttrOnce attr_once;
    if (smem > 48 * 1024) {
        int rc = attr_once.ensure(orientation_hist_pyr_kernel, smem, "orientation_hist_pyr smem attr");
        if (rc != AG_OK) return rc;
    }
    orientation_hist_pyr_kernel<<<cdiv(plan->B * cap, HCP_WARPS), HCP_WARPS * 32, smem, (cudaStream_t)stream>>>(
        P, d_pyr, d_lafs, d_oct, d_lvl, d_count, cap, PS, d_angle, d_lafs_out);
    AG_CHECK_LAUNCH("orientation_hist_pyr_kernel");
    return AG_OK;
}

int ag_baumberg_shape_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct, const int* d_lvl,
                          const int* d_count, int cap, int PS, int n_iters, float* d_A, void* stream) {
    AG_REQUIRE(plan && d_pyr && d_lafs && d_oct && d_lvl && d_A, "NULL argument");
    AG_REQUIRE(PS >= 3 && PS <= HC_MAXPS, "patch size out of range (3..41)");
    AG_REQUIRE(n_iters >= 1 && n_iters <= 64, "n_iters out of range (1..64)");
    AG_REQUIRE(cap >= 1 && (long long)plan->B * cap <= (1ll << 30), "bad sizes");
    HcPyrArgs P;
    hcp_args(plan, PS, (PS / 2.0) / 3.0, 1.0f, P);   // AffineShapeEstimator: CircularGaussKernel(PS, sigma = PS/2/3)
    const size_t smem = hcp_smem_bytes(PS, false);
    static SmemAttrOnce attr_once;
    if (smem > 48 * 1024) {
        int rc = attr_once.ensure(baumberg_pyr_kernel, smem, "baumberg_pyr smem attr");
        if (rc != AG_OK) return rc;
    }
    baumberg_pyr_kernel<<<cdiv(plan->B * cap, HCP_WARPS), HCP_WARPS * 32, smem, (cudaStream_t)stream>>>(
        P, d_pyr, d_lafs, d_oct, d_lvl, d_count, cap, PS, n_iters, d_A);
    AG_CHECK_LAUNCH("baumberg_pyr_kernel");
    return AG_OK;
}

}  // extern "C"
