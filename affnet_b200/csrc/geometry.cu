// Per-keypoint geometry: affine-shape filter, orientation compose, LAF (de)normalisation
// (SURVEY.md §8a rows a10 (partly), a11, a13, a14).
//
// Replaces the tail of getAffineShape (SparseImgRepresenter.py:136-162) with batch_eig2x2 (Utils.py:168-175)
// and checkTouchBoundary (LAF.py:98-104), the compose step of getOrientation (SparseImgRepresenter.py:175)
// and denormalizeLAFs / normalizeLAFs (LAF.py:407-429).
// Decisions (eigen-ratio test, boundary test) use the reference's fp32 operation order with non-contracted
// intrinsics so that identical A matrices give the identical survivor set.
#include "common.cuh"

namespace ag {

constexpr int GNT = 1024;

struct ShapeParams {
    const float* A;      // [B,cap,2,2]
    const float* resp;   // [B,cap]
    const float* lafs;   // [B,cap,2,3]
    const int* oct;
    const int* lvl;
    const int* count_in;
    int cap, num_features, out_cap, sort_cap;
    float* resp_out;
    float* lafs_out;
    int* oct_out;
    int* lvl_out;
    int* count_out;
};

__device__ __forceinline__ bool shape_ok(const float* A, const float* NL) {
    // batch_eig2x2 (Utils.py:168-175)
    const float trace = __fadd_rn(A[0], A[3]);
    const float det = __fsub_rn(__fmul_rn(A[0], A[3]), __fmul_rn(A[2], A[1]));
    const float delta1 = __fsub_rn(__fmul_rn(trace, trace), __fmul_rn(4.0f, det));
    float l1, l2;
    if (delta1 > 0.f) {
        const float delta = __fsqrt_rn(fabsf(delta1));
        l1 = __fdiv_rn(__fadd_rn(trace, delta), 2.0f);
        l2 = __fdiv_rn(__fsub_rn(trace, delta), 2.0f);
    } else {
        l1 = 1000.0f; l2 = 0.0001f;
    }
    const float ratio = fabsf(__fdiv_rn(l1, __fadd_rn(l2, 1e-8f)));
    bool ok = (ratio < 6.0f) && (ratio > (float)(1.0 / 6.0));  // SparseImgRepresenter.py:149
    // checkTouchBoundary (LAF.py:98-104): corners (+-1,+-1) through the normalised LAF must lie in [0,1] (Q5)
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const float x = (c & 2) ? 1.f : -1.f, y = (c & 1) ? 1.f : -1.f;
        const float ox = fmaf(NL[0], x, fmaf(NL[1], y, NL[2]));
        const float oy = fmaf(NL[3], x, fmaf(NL[4], y, NL[5]));
        ok = ok && !(ox > 1.0f || ox < 0.0f || oy > 1.0f || oy < 0.0f);
    }
    return ok;
}

__device__ __forceinline__ void compose_laf(const float* A, const float* L, float* NL) {
    // new_LAF = [bmm(A, LAF[:, :, 0:2]), LAF[:, :, 2:]]   SparseImgRepresenter.py:138
    NL[0] = fmaf(A[0], L[0], A[1] * L[3]); NL[1] = fmaf(A[0], L[1], A[1] * L[4]); NL[2] = L[2];
    NL[3] = fmaf(A[2], L[0], A[3] * L[3]); NL[4] = fmaf(A[2], L[1], A[3] * L[4]); NL[5] = L[5];
}

__global__ void __launch_bounds__(GNT) shape_filter_kernel(const ShapeParams P) {
    extern __shared__ unsigned long long s_key[];
    __shared__ int s_surv;
    const int b = blockIdx.x;
    const int n = max(0, min(P.count_in[b], P.cap));
    const float* A = P.A + (size_t)b * P.cap * 4;
    const float* L = P.lafs + (size_t)b * P.cap * 6;
    const float* R = P.resp + (size_t)b * P.cap;
    if (threadIdx.x == 0) s_surv = 0;
    __syncthreads();
    // pass 1: count survivors
    int local = 0;
    for (int i = threadIdx.x; i < n; i += GNT) {
        float NL[6];
        compose_laf(A + i * 4, L + i * 6, NL);
        local += shape_ok(A + i * 4, NL) ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(&s_surv, local);
    __syncthreads();
    const int S = s_surv;
    const bool sorted = (P.num_features > 0) && (S > P.num_features);  // SparseImgRepresenter.py:151
    int m = sorted ? P.num_features : S;
    if (m > P.out_cap) m = P.out_cap;
    // pass 2: keys
    for (int i = threadIdx.x; i < P.sort_cap; i += GNT) {
        unsigned long long k = 0ull;
        if (i < n) {
            float NL[6];
            compose_laf(A + i * 4, L + i * 6, NL);
            const bool ok = shape_ok(A + i * 4, NL);
            const unsigned hi = sorted ? float_to_ordered(ok ? R[i] : 0.f) : (ok ? 1u : 0u);
            k = ((unsigned long long)hi << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i);
        }
        s_key[i] = k;
    }
    __syncthreads();
    bitonic_sort_desc<false>(s_key, nullptr, P.sort_cap);
    for (int r = threadIdx.x; r < m; r += GNT) {
        const int i = (int)(0xFFFFFFFFu - (unsigned)(s_key[r] & 0xFFFFFFFFull));
        const size_t o = (size_t)b * P.out_cap + r;
        float NL[6];
        compose_laf(A + i * 4, L + i * 6, NL);
        P.resp_out[o] = R[i];
#pragma unroll
        for (int q = 0; q < 6; q++) P.lafs_out[o * 6 + q] = NL[q];
        P.oct_out[o] = P.oct[(size_t)b * P.cap + i];
        P.lvl_out[o] = P.lvl[(size_t)b * P.cap + i];
    }
    if (threadIdx.x == 0) P.count_out[b] = (P.count_in[b] < 0) ? -1 : m;   // -1 = upstream capacity overflow, propagated
}

__global__ void lafs_rotate_kernel(float* __restrict__ lafs, const float* __restrict__ R, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float* L = lafs + (size_t)i * 6;
    const float* r = R + (size_t)i * 4;
    float l[6] = {L[0], L[1], 0.f, L[3], L[4], 0.f};
    laf_rotate(l, r[0], r[1], r[2], r[3]);
    L[0] = l[0]; L[1] = l[1]; L[3] = l[3]; L[4] = l[4];
}

__global__ void lafs_scale_kernel(const float* __restrict__ in, float* __restrict__ out, int n, float ac, float xc, float yc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* L = in + (size_t)i * 6;
    float* O = out + (size_t)i * 6;
    O[0] = __fmul_rn(L[0], ac); O[1] = __fmul_rn(L[1], ac); O[2] = __fmul_rn(L[2], xc);
    O[3] = __fmul_rn(L[3], ac); O[4] = __fmul_rn(L[4], ac); O[5] = __fmul_rn(L[5], yc);
}

// LAFs2ellT (LAF.py:35-51) with the closed-form 2x2 SVD of bsvd2x2 (LAF.py:106-144): one thread per keypoint.  Only U and
// the singular values of A / scale enter the result: ell = (x, y, M00, M01, M11), M = U diag(1 / (scale^2 s_i^2)) U^T.
__global__ void lafs_to_ell_kernel(const float* __restrict__ lafs, float* __restrict__ ell, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* L = lafs + (size_t)i * 6;
    const float scale = sqrtf(L[0] * L[4] - L[1] * L[3] + 1e-10f);
    const float a00 = L[0] / scale, a01 = L[1] / scale, a10 = L[3] / scale, a11 = L[4] / scale;
    // Su = A A^T
    const float s00 = a00 * a00 + a01 * a01, s01 = a00 * a10 + a01 * a11, s11 = a10 * a10 + a11 * a11;
    const float phi = 0.5f * atan2f(s01 + s01 + 1e-12f, s00 - s11 + 1e-12f);
    const float c = cosf(phi), sn = sinf(phi);   // U = [[c, -s], [s, c]]
    const float sum = s00 + s11;
    const float dif = sqrtf((s00 - s11) * (s00 - s11) + 4.0f * s01 * s01 + 1e-12f);
    const float sig0 = sqrtf((sum + dif) / 2.0f), sig1 = sqrtf((sum - dif) / 2.0f);
    const float w0 = 1.0f / (scale * scale * sig0 * sig0), w1 = 1.0f / (scale * scale * sig1 * sig1);
    float* o = ell + (size_t)i * 5;
    o[0] = L[2]; o[1] = L[5];
    o[2] = c * w0 * c + sn * w1 * sn;          // (U W U^T)[0][0]
    o[3] = c * w0 * sn - sn * w1 * c;          // [0][1]
    o[4] = sn * w0 * sn + c * w1 * c;          // [1][1]
}

}  // namespace ag

using namespace ag;

namespace ag {
// out = A * B for [n,2,2] batches, in torch.bmm's fp32 operation order (row-by-column, two products added left to right): the Baumberg
// chain base_A <- A base_A of SparseImgRepresenter.py:133
__global__ void mat2_compose_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float a[4] = {A[i * 4], A[i * 4 + 1], A[i * 4 + 2], A[i * 4 + 3]};
    const float b[4] = {B[i * 4], B[i * 4 + 1], B[i * 4 + 2], B[i * 4 + 3]};
    float o[4];
    mat2_mul(a, b, o);
#pragma unroll
    for (int q = 0; q < 4; q++) out[i * 4 + q] = o[q];
}
// out = [A * L[:, :, :2] | L[:, :, 2]] : the working LAF of the next Baumberg iteration (SparseImgRepresenter.py:134-135)
__global__ void lafs_left_multiply_kernel(const float* __restrict__ A, const float* __restrict__ Lf, float* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float a[4] = {A[i * 4], A[i * 4 + 1], A[i * 4 + 2], A[i * 4 + 3]};
    const float l[6] = {Lf[i * 6], Lf[i * 6 + 1], Lf[i * 6 + 2], Lf[i * 6 + 3], Lf[i * 6 + 4], Lf[i * 6 + 5]};
    float o[6];
    laf_left_mul(a, l, o);
#pragma unroll
    for (int q = 0; q < 6; q++) out[i * 6 + q] = o[q];
}
}  // namespace ag

extern "C" {

int ag_affine_shape_filter(const float* d_A, const float* d_resp, const float* d_lafs, const int* d_oct, const int* d_lvl,
                           const int* d_count_in, int B, int cap, int num_features, int out_cap, float* d_resp_out,
                           float* d_lafs_out, int* d_oct_out, int* d_lvl_out, int* d_count_out, void* stream) {
    AG_REQUIRE(d_A && d_resp && d_lafs && d_oct && d_lvl && d_count_in && d_resp_out && d_lafs_out && d_oct_out &&
                   d_lvl_out && d_count_out, "NULL argument");
    AG_REQUIRE(B >= 1 && cap >= 1 && out_cap >= 1, "bad sizes");
    int sort_cap = 32;
    while (sort_cap < cap) sort_cap <<= 1;
    const size_t smem = (size_t)sort_cap * sizeof(unsigned long long);
    if (smem > 200 * 1024) {
        set_error("ag_affine_shape_filter: cap %d needs %zu B of shared memory (max 200 KiB)", cap, smem);
        return AG_ERR_CAPACITY;
    }
    static SmemAttrOnce attr_once;
    if (smem > 32 * 1024) {  // static + dynamic must stay under the 48 KiB default
        int rc = attr_once.ensure(shape_filter_kernel, smem, "shape smem attr");
        if (rc != AG_OK) return rc;
    }
    ShapeParams P;
    P.A = d_A; P.resp = d_resp; P.lafs = d_lafs; P.oct = d_oct; P.lvl = d_lvl; P.count_in = d_count_in;
    P.cap = cap; P.num_features = num_features; P.out_cap = out_cap; P.sort_cap = sort_cap;
    P.resp_out = d_resp_out; P.lafs_out = d_lafs_out; P.oct_out = d_oct_out; P.lvl_out = d_lvl_out; P.count_out = d_count_out;
    shape_filter_kernel<<<B, GNT, smem, (cudaStream_t)stream>>>(P);
    AG_CHECK_LAUNCH("shape_filter_kernel");
    return AG_OK;
}

int ag_lafs_apply_rotation(float* d_lafs, const float* d_R, int n, void* stream) {
    AG_REQUIRE(d_lafs && d_R, "NULL argument");
    if (n <= 0) return AG_OK;
    lafs_rotate_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_lafs, d_R, n);
    AG_CHECK_LAUNCH("lafs_rotate_kernel");
    return AG_OK;
}

int ag_mat2_compose(const float* d_A, const float* d_B, float* d_out, int n, void* stream) {
    AG_REQUIRE(d_A && d_B && d_out, "NULL argument");
    if (n <= 0) return AG_OK;
    mat2_compose_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_A, d_B, d_out, n);
    AG_CHECK_LAUNCH("mat2_compose_kernel");
    return AG_OK;
}

int ag_lafs_left_multiply(const float* d_A, const float* d_lafs, float* d_out, int n, void* stream) {
    AG_REQUIRE(d_A && d_lafs && d_out, "NULL argument");
    if (n <= 0) return AG_OK;
    lafs_left_multiply_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_A, d_lafs, d_out, n);
    AG_CHECK_LAUNCH("lafs_left_multiply_kernel");
    return AG_OK;
}

int ag_lafs_scale(const float* d_in, float* d_out, int n, float a_coef, float x_coef, float y_coef, void* stream) {
    AG_REQUIRE(d_in && d_out, "NULL argument");
    if (n <= 0) return AG_OK;
    lafs_scale_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_in, d_out, n, a_coef, x_coef, y_coef);
    AG_CHECK_LAUNCH("lafs_scale_kernel");
    return AG_OK;
}

int ag_lafs_to_ell(const float* d_lafs, int n, float* d_ell, void* stream) {
    AG_REQUIRE(d_lafs && d_ell, "NULL argument");
    if (n <= 0) return AG_OK;
    lafs_to_ell_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_lafs, d_ell, n);
    AG_CHECK_LAUNCH("lafs_to_ell_kernel");
    return AG_OK;
}

}  // extern "C"
