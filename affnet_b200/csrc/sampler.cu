// Affine bilinear patch sampler and pyramid-level routing (SURVEY.md §8a rows a7, a8, a15).
//
// Replaces generate_patch_grid_from_normalized_LAFs + extract_patches + batched_grid_apply
// (LAF.py:313-372: F.affine_grid + F.grid_sample, bilinear, zeros padding, align_corners=False),
// extract_patches_from_pyramid_with_inv_index / get_inverted_pyr_index (LAF.py:376-404) and
// get_pyramid_and_level_index_for_LAFs (LAF.py:450-472).
//
// Closed form: out[n,c,i,j] = bilinear(img_c, p - 0.5),  p = A_px (x_j, y_i)^T + t_px,
// x_j = (2j+1)/PS - 1, A_px = LAF_A * min(h,w), t_px = (LAF_x * w, LAF_y * h).
// The (octave, level) bucketing of the reference (nonzero + scatter) is replaced by direct per-keypoint
// routing: one warp-row of threads per patch row reads its own level of the L2-resident pyramid.
#include "common.cuh"

namespace ag {

__global__ void extract_patches_kernel(const float* __restrict__ img, int C, int h, int w, int per_patch_img,
                                       const float* __restrict__ lafs, int n, int PS, float* __restrict__ out) {
    const int pi = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= PS * PS) return;
    const int i = t / PS, j = t - i * PS;
    float px, py;
    laf_sample_xy(lafs + (size_t)pi * 6, h, w, i, j, 1.0f / (float)PS, px, py);
    const float* base = img + (per_patch_img ? (size_t)pi * C * h * w : 0);
    for (int c = 0; c < C; c++)
        out[((size_t)pi * C + c) * PS * PS + t] = bilinear_zero(base + (size_t)c * h * w, h, w, px, py);
}

__global__ void extract_patches_pyr_kernel(const PyrGeom G, const float* __restrict__ pyr, const float* __restrict__ lafs,
                                           const int* __restrict__ oct, const int* __restrict__ lvl,
                                           const int* __restrict__ count, int cap, int PS, float* __restrict__ out) {
    const int b = blockIdx.z, pi = blockIdx.y;
    if (count != nullptr && pi >= count[b]) return;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= PS * PS) return;
    const size_t row = (size_t)b * cap + pi;
    const int o = clampi(oct[row], 0, G.n_octaves - 1), l = clampi(lvl[row], 0, G.n_levels - 1);
    const int h = G.h[o], w = G.w[o];
    const float* img = pyr + G.off[o][l] + (size_t)b * h * w;
    const int i = t / PS, j = t - i * PS;
    float px, py;
    laf_sample_xy(lafs + row * 6, h, w, i, j, 1.0f / (float)PS, px, py);
    out[row * PS * PS + t] = bilinear_zero(img, h, w, px, py);
}

struct LevelCands {
    int n;
    double cand[AG_MAX_OCTAVES * AG_MAX_LEVELS];
    unsigned char oct[AG_MAX_OCTAVES * AG_MAX_LEVELS], lvl[AG_MAX_OCTAVES * AG_MAX_LEVELS];
};

__global__ void level_for_lafs_kernel(const LevelCands C, const float* __restrict__ dlafs, int n, float PS,
                                      int* __restrict__ oct, int* __restrict__ lvl) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* L = dlafs + (size_t)i * 6;
    // get_LAFs_scales (LAF.py:450-451): fp32, separate products
    const float det = __fsub_rn(__fmul_rn(L[0], L[4]), __fmul_rn(L[1], L[3]));
    const float scale = __fsqrt_rn(__fadd_rn(fabsf(det), 1e-12f));
    const double needed = (double)__fdiv_rn(scale, PS);
    int best = 0;
    double bd = fabs(C.cand[0] - needed);
    for (int k = 1; k < C.n; k++) {
        const double d = fabs(C.cand[k] - needed);
        if (d < bd) { bd = d; best = k; }  // first minimum wins (numpy argmin)
    }
    oct[i] = C.oct[best];
    lvl[i] = C.lvl[best];
}

}  // namespace ag

using namespace ag;

extern "C" {

int ag_extract_patches(const float* d_img, int C, int h, int w, int per_patch_img, const float* d_lafs, int n, int PS,
                       float* d_out, void* stream) {
    AG_REQUIRE(d_img && d_lafs && d_out, "NULL argument");
    AG_REQUIRE(C >= 1 && h >= 1 && w >= 1 && PS >= 1 && n >= 0, "bad sizes");
    if (n == 0) return AG_OK;
    AG_REQUIRE(n <= 65535 * 1, "n too large for one launch (max 65535)");
    dim3 grid(cdiv(PS * PS, 256), n);
    extract_patches_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_img, C, h, w, per_patch_img, d_lafs, n, PS, d_out);
    AG_CHECK_LAUNCH("extract_patches_kernel");
    return AG_OK;
}

int ag_extract_patches_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                           const int* d_lvl, const int* d_count, int cap, int PS, float* d_out, void* stream) {
    AG_REQUIRE(plan && d_pyr && d_lafs && d_oct && d_lvl && d_out, "NULL argument");
    AG_REQUIRE(cap >= 1 && cap <= 65535 && PS >= 1, "bad sizes");
    dim3 grid(cdiv(PS * PS, 256), cap, plan->B);
    extract_patches_pyr_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(make_geom(plan), d_pyr, d_lafs, d_oct, d_lvl, d_count,
                                                                        cap, PS, d_out);
    AG_CHECK_LAUNCH("extract_patches_pyr_kernel");
    return AG_OK;
}

int ag_pyramid_level_for_lafs(const ag_pyramid_plan_t* plan, const float* d_dlafs, int n, int PS, int* d_oct, int* d_lvl,
                              void* stream) {
    AG_REQUIRE(plan && d_dlafs && d_oct && d_lvl, "NULL argument");
    if (n <= 0) return AG_OK;
    LevelCands C;
    C.n = 0;
    for (int o = 0; o < plan->n_octaves; o++)
        for (int l = 0; l < plan->n_levels; l++) {  // octave-major, LAF.py:458-461
            C.cand[C.n] = plan->sigma[o][l] * plan->pix_dist[o];
            C.oct[C.n] = (unsigned char)o; C.lvl[C.n] = (unsigned char)l;
            C.n++;
        }
    level_for_lafs_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(C, d_dlafs, n, (float)PS, d_oct, d_lvl);
    AG_CHECK_LAUNCH("level_for_lafs_kernel");
    return AG_OK;
}

}  // extern "C"
