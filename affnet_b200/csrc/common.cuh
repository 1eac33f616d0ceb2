// Shared helpers for the affnet_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/affnet_b200.h"

namespace ag {

void set_error(const char* fmt, ...);
extern thread_local int g_launches;  // kernels launched since last reset (host-side counter)

inline int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return AG_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return (e == cudaErrorNoKernelImageForDevice || e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver)
               ? AG_ERR_NO_DEVICE
               : AG_ERR_CUDA;
}

void prof_mark(const char* name);  // records an event after a launch when profiling is on (see ag_prof_begin)

#define AG_CHECK_LAUNCH(name)                                        \
    do {                                                             \
        ::ag::g_launches++;                                          \
        int _rc = ::ag::check_cuda(cudaGetLastError(), name);        \
        if (_rc != AG_OK) return _rc;                                \
        ::ag::prof_mark(name);                                       \
    } while (0)

#define AG_REQUIRE(cond, msg)                                        \
    do {                                                             \
        if (!(cond)) {                                               \
            ::ag::set_error("%s: %s", __func__, msg);                \
            return AG_ERR_INVALID;                                   \
        }                                                            \
    } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember per device what was set (a process may drive several GPUs)
struct SmemAttrOnce {
    size_t set[64] = {};
    template <typename K>
    int ensure(K kernel, size_t bytes, const char* what) {
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 63;
        if (bytes <= set[dev]) return AG_OK;
        int rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), what);
        if (rc == AG_OK) set[dev] = bytes;
        return rc;
    }
};

inline int cdiv(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Order-preserving float -> uint32 (larger float => larger uint), total order incl. negatives.
__host__ __device__ inline uint32_t float_to_ordered(float f) {
    uint32_t u;
#ifdef __CUDA_ARCH__
    u = __float_as_uint(f);
#else
    memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Block-wide bitonic sort (descending) of n = 2^k 64-bit keys in shared memory, optionally with an int payload.  Every thread owns whole
// compare-exchange PAIRS (pair p -> elements i = p with a 0 bit inserted at log2(j), i | j), so no thread idles on the "ixj > i" half:
// half the loop trips of the textbook form (select_kernel: 163 -> ~95 us for 4096 keys on 1024 threads).
template <bool HAS_IDX>
__device__ __forceinline__ void bitonic_sort_desc(unsigned long long* key, int* idx, int n) {
    for (int k2 = 2; k2 <= n; k2 <<= 1)
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int p = threadIdx.x; p < (n >> 1); p += blockDim.x) {
                const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), l = i | j;
                const unsigned long long a = key[i], c = key[l];
                const bool desc = (i & k2) == 0;
                if (desc ? (a < c) : (a > c)) {
                    key[i] = c; key[l] = a;
                    if (HAS_IDX) { const int t = idx[i]; idx[i] = idx[l]; idx[l] = t; }
                }
            }
            __syncthreads();
        }
}

// Bilinear tap with zeros outside the image (F.grid_sample, padding_mode='zeros').  Explicit rounding steps so that the
// standalone sampler and the sampler fused into the first CNN layer produce identical bits.
__device__ __forceinline__ float bilinear_zero(const float* __restrict__ img, int h, int w, float px, float py) {
    const float fx0 = floorf(px), fy0 = floorf(py);
    const int x0 = (int)fx0, y0 = (int)fy0;
    const float ax = __fsub_rn(px, fx0), ay = __fsub_rn(py, fy0);
    const float bx = __fsub_rn(1.f, ax), by = __fsub_rn(1.f, ay);
    const bool xin0 = (x0 >= 0) & (x0 < w), xin1 = (x0 + 1 >= 0) & (x0 + 1 < w);
    const bool yin0 = (y0 >= 0) & (y0 < h), yin1 = (y0 + 1 >= 0) & (y0 + 1 < h);
    const float v00 = (xin0 & yin0) ? __ldg(img + (size_t)y0 * w + x0) : 0.f;
    const float v01 = (xin1 & yin0) ? __ldg(img + (size_t)y0 * w + x0 + 1) : 0.f;
    const float v10 = (xin0 & yin1) ? __ldg(img + (size_t)(y0 + 1) * w + x0) : 0.f;
    const float v11 = (xin1 & yin1) ? __ldg(img + (size_t)(y0 + 1) * w + x0 + 1) : 0.f;
    const float top = __fmaf_rn(v01, ax, __fmul_rn(v00, bx)), bot = __fmaf_rn(v11, ax, __fmul_rn(v10, bx));
    return __fmaf_rn(bot, ay, __fmul_rn(top, by));
}

// The same tap in two phases (issue the four loads early, combine later); bit-identical to bilinear_zero.
__device__ __forceinline__ void bilinear_taps(const float* __restrict__ img, int h, int w, float px, float py, float (&t)[4], float& ax, float& ay) {
    const float fx0 = floorf(px), fy0 = floorf(py);
    const int x0 = (int)fx0, y0 = (int)fy0;
    ax = __fsub_rn(px, fx0); ay = __fsub_rn(py, fy0);
    const bool xin0 = (x0 >= 0) & (x0 < w), xin1 = (x0 + 1 >= 0) & (x0 + 1 < w);
    const bool yin0 = (y0 >= 0) & (y0 < h), yin1 = (y0 + 1 >= 0) & (y0 + 1 < h);
    t[0] = (xin0 & yin0) ? __ldg(img + (size_t)y0 * w + x0) : 0.f;
    t[1] = (xin1 & yin0) ? __ldg(img + (size_t)y0 * w + x0 + 1) : 0.f;
    t[2] = (xin0 & yin1) ? __ldg(img + (size_t)(y0 + 1) * w + x0) : 0.f;
    t[3] = (xin1 & yin1) ? __ldg(img + (size_t)(y0 + 1) * w + x0 + 1) : 0.f;
}
__device__ __forceinline__ float bilinear_combine(const float (&t)[4], float ax, float ay) {
    const float bx = __fsub_rn(1.f, ax), by = __fsub_rn(1.f, ay);
    const float top = __fmaf_rn(t[1], ax, __fmul_rn(t[0], bx)), bot = __fmaf_rn(t[3], ax, __fmul_rn(t[2], bx));
    return __fmaf_rn(bot, ay, __fmul_rn(top, by));
}

// Patch-grid coordinate of sample (i,j) of a PSxPS patch under a normalised LAF on an h x w image (LAF.py:313-324).
__device__ __forceinline__ void laf_sample_xy(const float* __restrict__ L, int h, int w, int i, int j, float inv_ps, float& px, float& py) {
    const float ms = (float)min(h, w);
    const float a11 = __fmul_rn(L[0], ms), a12 = __fmul_rn(L[1], ms), tx = __fmul_rn(L[2], (float)w);
    const float a21 = __fmul_rn(L[3], ms), a22 = __fmul_rn(L[4], ms), ty = __fmul_rn(L[5], (float)h);
    const float xj = __fsub_rn(__fmul_rn(__fmaf_rn(2.f, (float)j, 1.f), inv_ps), 1.f), yi = __fsub_rn(__fmul_rn(__fmaf_rn(2.f, (float)i, 1.f), inv_ps), 1.f);
    px = __fsub_rn(__fmaf_rn(a11, xj, __fmaf_rn(a12, yi, tx)), 0.5f);
    py = __fsub_rn(__fmaf_rn(a21, xj, __fmaf_rn(a22, yi, ty)), 0.5f);
}

// Pyramid geometry passed by value to the kernels that sample patches straight from the pyramid (row b*cap+i reads level
// pyr[oct][lvl] of image b).
struct PyrGeom {
    int n_octaves, n_levels, B;
    int h[AG_MAX_OCTAVES], w[AG_MAX_OCTAVES];
    long long off[AG_MAX_OCTAVES][AG_MAX_LEVELS];
};

inline PyrGeom make_geom(const ag_pyramid_plan_t* p) {
    PyrGeom g;
    g.n_octaves = p->n_octaves; g.n_levels = p->n_levels; g.B = p->B;
    for (int o = 0; o < AG_MAX_OCTAVES; o++) {
        g.h[o] = p->h[o]; g.w[o] = p->w[o];
        for (int l = 0; l < AG_MAX_LEVELS; l++) g.off[o][l] = p->level_offset[o][l];
    }
    return g;
}

// LAF_A <- LAF_A * R for R = [r0 r1; r2 r3] (getOrientation's compose, SparseImgRepresenter.py:175)
__device__ __forceinline__ void laf_rotate(float (&l)[6], float r0, float r1, float r2, float r3) {
    const float l00 = l[0], l01 = l[1], l10 = l[3], l11 = l[4];
    l[0] = fmaf(l00, r0, l01 * r2); l[1] = fmaf(l00, r1, l01 * r3);
    l[3] = fmaf(l10, r0, l11 * r2); l[4] = fmaf(l10, r1, l11 * r3);
}

// out = a * b for 2x2 matrices, in torch.bmm's fp32 operation order (row-by-column, two products added left to right)
__device__ __forceinline__ void mat2_mul(const float (&a)[4], const float (&b)[4], float (&out)[4]) {
    out[0] = __fmaf_rn(a[1], b[2], __fmul_rn(a[0], b[0])); out[1] = __fmaf_rn(a[1], b[3], __fmul_rn(a[0], b[1]));
    out[2] = __fmaf_rn(a[3], b[2], __fmul_rn(a[2], b[0])); out[3] = __fmaf_rn(a[3], b[3], __fmul_rn(a[2], b[1]));
}

// out = [a * l[:, :2] | l[:, 2]] for a 2x2 matrix a and a LAF l (the bmm of SparseImgRepresenter.py:134-135)
__device__ __forceinline__ void laf_left_mul(const float (&a)[4], const float (&l)[6], float (&out)[6]) {
    out[0] = __fmaf_rn(a[1], l[3], __fmul_rn(a[0], l[0])); out[1] = __fmaf_rn(a[1], l[4], __fmul_rn(a[0], l[1])); out[2] = l[2];
    out[3] = __fmaf_rn(a[3], l[3], __fmul_rn(a[2], l[0])); out[4] = __fmaf_rn(a[3], l[4], __fmul_rn(a[2], l[1])); out[5] = l[5];
}

}  // namespace ag
