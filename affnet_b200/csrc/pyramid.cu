// Gaussian scale-space pyramid (SURVEY.md §8a rows a1, a2).
//
// Replaces ScalePyramid.forward (HandCraftedModules.py:13-56) and GaussianBlur (Utils.py:92-114,150-166).
// The reference convolves with a dense k x k kernel that is an exact outer product (Q1), so each blur
// is done here as a fused horizontal+vertical separable pass through shared memory: one HBM/L2 read of
// the source tile (+halo), one write of the blurred tile, and - for the level that seeds the next
// octave - the stride-2 decimated copy (F.avg_pool2d(k=1, s=2)) from the same registers.
#include <math.h>
#include <stdarg.h>

#include <string>
#include <vector>

#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, libcuda is not linked)

#include "common.cuh"

namespace ag {

static thread_local char g_err[512] = "";
thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---- per-launch CUDA-event profiler (bench.py's roofline leg) ---------------------------------------
struct Prof {
    bool on = false;
    cudaStream_t st = nullptr;
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> names;
    std::vector<float> ms;
};
static Prof g_prof;

void prof_mark(const char* name) {
    if (!g_prof.on) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, g_prof.st);
    g_prof.ev.push_back(e);
    g_prof.names.push_back(name);
}

// ---- host: kernel taps exactly as CircularGaussKernel builds them (float64 -> float32) -------------
constexpr int kMaxRadius = 12;  // sigma up to ~4.0
struct BlurTaps {
    int r;
    float w[2 * kMaxRadius + 1];
};

int gauss_kernel_size(double sigma) {  // Utils.py:95-97
    int k = (int)(2.0 * 3.0 * sigma + 1.0);
    if (k % 2 == 0) k += 1;
    return k;
}

int make_taps(double sigma, BlurTaps* t) {
    int k = gauss_kernel_size(sigma);
    if (k < 1 || k > 2 * kMaxRadius + 1) {
        set_error("gaussian sigma %.4f needs %d taps (max %d)", sigma, k, 2 * kMaxRadius + 1);
        return AG_ERR_INVALID;
    }
    // Utils.py:98-113 under python3: halfSize = k/2 (true division), x = linspace(-half, half, k)
    double half = k / 2.0, e[2 * kMaxRadius + 1], sum = 0.0;
    double step = (k > 1) ? (2.0 * half) / (k - 1) : 0.0;
    for (int i = 0; i < k; i++) {
        double x = (i == k - 1) ? half : -half + i * step;
        e[i] = exp(-(x * x) / (2.0 * sigma * sigma));
        sum += e[i];
    }
    t->r = k / 2;
    for (int i = 0; i < k; i++) t->w[i] = (float)(e[i] / sum);
    return AG_OK;
}

// ---- device: fused separable blur ---------------------------------------------------------------
// 64x64 output tile per CTA.  Both passes are register blocked so that shared memory is read with 128-bit loads:
//   horizontal: one thread -> 4 adjacent outputs of a row from 4+2R inputs (ceil((4+2R)/4) LDS.128, 4*(2R+1) FMA)
//   vertical  : one thread -> 4x4 outputs (4 rows of a column quad) from 4+2R rows of the intermediate (4+2R LDS.128)
// The tile is written with 128-bit stores when the row pitch allows it, and the stride-2 decimated copy that seeds the next
// octave (F.avg_pool2d(k=1, s=2), HandCraftedModules.py:47) comes from the same registers.
constexpr int TW = 64, TH = 64, NT = 256;

template <int R>
struct BlurGeom {
    static constexpr int IH = TH + 2 * R;                      // rows of the input window
    static constexpr int IWQ = (TW + 2 * R + 3) / 4 + 1;       // float4 per input row (window start aligned down to 4)
    static constexpr int IW = IWQ * 4;
    static constexpr int NQ = (4 + 2 * R + 3) / 4 + 1;         // float4 a horizontal quad may touch (window start not aligned)
    static constexpr size_t SMEM = sizeof(float) * ((size_t)IH * IW + (size_t)IH * TW);
};

template <int R>
__global__ void __launch_bounds__(NT) blur_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                   float* __restrict__ dec, int h, int w, BlurTaps taps,
                                                   const __grid_constant__ CUtensorMap tmap, int use_tmap) {
    using G = BlurGeom<R>;
    extern __shared__ __align__(128) float smem_f[];
    float* s_in = smem_f;                       // [IH][IW]; column c holds image column x0 - R4 + c, R4 = R rounded up to 4
    float* s_mid = smem_f + G::IH * G::IW;      // [IH][TW]
    constexpr int R4 = (R + 3) / 4 * 4;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const float* img = in + (size_t)b * h * w;
    // 1. input window with replicate (clamp) addressing
#ifndef AG_BLUR_SCALAR_FILL
    // interior tiles: same values in the same places as the clamped fill below, so the arithmetic does not change
    const bool wide = (w & 3) == 0 && x0 - R4 >= 0 && x0 - R4 + G::IW <= w && (reinterpret_cast<size_t>(img) & 15) == 0;
#ifndef AG_BLUR_LDG_FILL
    // ... and tiles that need no row clamp either take the window as IH bulk copies (one 16-byte-aligned row segment each, completion
    // counted on one mbarrier): no thread spends issue slots or registers on moving the data
    __shared__ __align__(8) unsigned long long s_bar;
    const bool bulk = wide && y0 - R >= 0 && y0 - R + G::IH <= h;    // block-uniform
    if (bulk) {
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(G::IH * G::IW * 4)) : "memory");
        }
        __syncthreads();
        if (use_tmap) {
            // the whole window is ONE box of the level's tensor map [B][h][w] (TMA tile mode: IW x IH x 1 floats land densely = s_in's layout)
            if (threadIdx.x == 0)
                asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                                 (uint32_t)__cvta_generic_to_shared(s_in)),
                             "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(x0 - R4), "r"(y0 - R), "r"(b), "r"(bar)
                             : "memory");
        } else if ((threadIdx.x & 31) == 0) {     // one lane per warp issues every (NT/32)-th row: the bulk-copy instruction is warp-uniform, 8 issuers shorten the queue
            const float* src = img + (size_t)(y0 - R) * w + (x0 - R4);
            for (int ly = threadIdx.x >> 5; ly < G::IH; ly += NT / 32)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 (uint32_t)__cvta_generic_to_shared(s_in + ly * G::IW)),
                             "l"(src + (size_t)ly * w), "r"((uint32_t)(G::IW * 4)), "r"(bar)
                             : "memory");
        }
        // warp 0 alone polls the mbarrier (256 polling threads spent 18 % of the kernel's issue slots in the try_wait loop); the others
        // wait in the block barrier below, which orders their reads after warp 0's acquire
        if (threadIdx.x < 32)
            asm volatile("{\n .reg .pred P;\n W_%=:\n mbarrier.try_wait.parity.shared::cta.b64 P, [%0], 0;\n @P bra D_%=;\n bra W_%=;\n D_%=:\n}\n" ::"r"(bar) : "memory");
    } else
#endif
    // 128-bit loads (the scalar fill was 30 % of this kernel's stall samples)
    if (wide) {
        constexpr int QW = G::IW / 4;
        static_assert(G::IW % 4 == 0, "window rows are whole float4s");
        for (int i = threadIdx.x; i < G::IH * QW; i += NT) {
            const int ly = i / QW, q = i - ly * QW;
            const int gy = clampi(y0 + ly - R, 0, h - 1);
            reinterpret_cast<float4*>(s_in)[i] = __ldg(reinterpret_cast<const float4*>(img + (size_t)gy * w + (x0 - R4)) + q);
        }
    } else
#endif
    for (int i = threadIdx.x; i < G::IH * G::IW; i += NT) {
        const int ly = i / G::IW, lx = i - ly * G::IW;
        const int gy = clampi(y0 + ly - R, 0, h - 1), gx = clampi(x0 + lx - R4, 0, w - 1);
        s_in[i] = __ldg(img + (size_t)gy * w + gx);
    }
    __syncthreads();
    // 2. horizontal pass: quads of 4 outputs; inputs of output x live at columns (x + R4 - R) .. (x + R4 + R)
    for (int i = threadIdx.x; i < G::IH * (TW / 4); i += NT) {
        const int ly = i / (TW / 4), q = i - ly * (TW / 4);
        constexpr int OFF = R4 - R;                                // 0..3
        float v[G::NQ * 4];
        const float4* row = reinterpret_cast<const float4*>(s_in + ly * G::IW + q * 4);
#pragma unroll
        for (int j = 0; j < G::NQ; j++) {
            const float4 t = row[j];
            v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
        }
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k <= 2 * R; k++) {
            const float wk = taps.w[k];
            o.x = fmaf(wk, v[OFF + k], o.x); o.y = fmaf(wk, v[OFF + k + 1], o.y);
            o.z = fmaf(wk, v[OFF + k + 2], o.z); o.w = fmaf(wk, v[OFF + k + 3], o.w);
        }
        *reinterpret_cast<float4*>(s_mid + ly * TW + q * 4) = o;
    }
    __syncthreads();
    // 3. vertical pass: 4 rows x 4 columns per thread
    const int h2 = (h + 1) >> 1, w2 = (w + 1) >> 1;
    const bool vec_ok = (w & 3) == 0;
    {
        const int q = threadIdx.x & 15, rb = threadIdx.x >> 4;     // column quad 0..15, row block 0..15 (4 rows each)
        float4 acc[4];
#pragma unroll
        for (int r = 0; r < 4; r++) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 4 + 2 * R; k++) {
            const float4 t = *reinterpret_cast<const float4*>(s_mid + (rb * 4 + k) * TW + q * 4);
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const int tap = k - r;
                if (tap >= 0 && tap <= 2 * R) {
                    const float wk = taps.w[tap];
                    acc[r].x = fmaf(wk, t.x, acc[r].x); acc[r].y = fmaf(wk, t.y, acc[r].y);
                    acc[r].z = fmaf(wk, t.z, acc[r].z); acc[r].w = fmaf(wk, t.w, acc[r].w);
                }
            }
        }
        const int gx = x0 + q * 4;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int gy = y0 + rb * 4 + r;
            if (gy >= h || gx >= w) continue;
            float* orow = out + (size_t)b * h * w + (size_t)gy * w + gx;
            const float vals[4] = {acc[r].x, acc[r].y, acc[r].z, acc[r].w};
            if (vec_ok) {
                *reinterpret_cast<float4*>(orow) = acc[r];           // w % 4 == 0 -> gx + 3 < w and 16-byte aligned
            } else {
#pragma unroll
                for (int e = 0; e < 4; e++)
                    if (gx + e < w) orow[e] = vals[e];
            }
            if (dec != nullptr && (gy & 1) == 0) {
                float* drow = dec + (size_t)b * h2 * w2 + (size_t)(gy >> 1) * w2 + (gx >> 1);
                drow[0] = vals[0];
                if (gx + 2 < w) drow[1] = vals[2];
            }
        }
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point table (no link against libcuda); NULL when the driver has none
typedef CUresult (*TmapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TmapEncodeFn tmap_encoder() {
    static TmapEncodeFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        if (getenv("AG_BLUR_NO_TMA") == nullptr) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
                fn = reinterpret_cast<TmapEncodeFn>(p);
            else
                cudaGetLastError();
        }
    }
    return fn;
}

// tensor map of one pyramid level [B][h][w] fp32 with a box of iw x ih x 1 elements; false when the level cannot be described (then the
// kernel's row-by-row bulk copies are used)
static bool make_level_tmap(CUtensorMap* m, const float* base, int B, int h, int w, int iw, int ih) {
    TmapEncodeFn enc = tmap_encoder();
    if (enc == nullptr || (w & 3) != 0 || (reinterpret_cast<size_t>(base) & 15) != 0 || iw > 256 || ih > 256) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)w * 4, (cuuint64_t)w * h * 4};        // bytes, dimensions 1 and 2
    const cuuint32_t box[3] = {(cuuint32_t)iw, (cuuint32_t)ih, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int launch_blur(const float* in, float* out, float* dec, int B, int h, int w, double sigma, cudaStream_t st) {
    BlurTaps taps;
    int rc = make_taps(sigma, &taps);
    if (rc != AG_OK) return rc;
    dim3 grid(cdiv(w, TW), cdiv(h, TH), B), block(NT);
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    switch (taps.r) {
#define AG_BLUR_CASE(R)                                                                                                   \
    case R: {                                                                                                             \
        static SmemAttrOnce attr_once;                                                                                    \
        rc = attr_once.ensure(blur_kernel<R>, BlurGeom<R>::SMEM, "blur smem attr");                                       \
        if (rc != AG_OK) return rc;                                                                                       \
        const int use_tmap = make_level_tmap(&tmap, in, B, h, w, BlurGeom<R>::IW, BlurGeom<R>::IH) ? 1 : 0;                 \
        blur_kernel<R><<<grid, block, BlurGeom<R>::SMEM, st>>>(in, out, dec, h, w, taps, tmap, use_tmap);                  \
    } break;
        AG_BLUR_CASE(1) AG_BLUR_CASE(2) AG_BLUR_CASE(3) AG_BLUR_CASE(4) AG_BLUR_CASE(5) AG_BLUR_CASE(6)
        AG_BLUR_CASE(7) AG_BLUR_CASE(8) AG_BLUR_CASE(9) AG_BLUR_CASE(10) AG_BLUR_CASE(11) AG_BLUR_CASE(12)
#undef AG_BLUR_CASE
        default:
            set_error("unsupported blur radius %d", taps.r);
            return AG_ERR_INVALID;
    }
    AG_CHECK_LAUNCH("blur_kernel");
    return AG_OK;
}

__global__ void decimate_kernel(const float* __restrict__ in, float* __restrict__ out, int h, int w, int h2, int w2) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
    if (x < w2) out[(size_t)b * h2 * w2 + (size_t)y * w2 + x] = in[(size_t)b * h * w + (size_t)(2 * y) * w + 2 * x];
}

}  // namespace ag

using namespace ag;

extern "C" {

const char* ag_last_error(void) { return ag::g_err; }
int ag_abi_version(void) { return 1; }

int ag_prof_begin(void* stream) {
    for (cudaEvent_t e : g_prof.ev) cudaEventDestroy(e);
    g_prof.ev.clear(); g_prof.names.clear(); g_prof.ms.clear();
    g_prof.st = (cudaStream_t)stream;
    g_prof.on = true;
    prof_mark("<begin>");
    return AG_OK;
}

int ag_prof_end(void) {
    g_prof.on = false;
    if (g_prof.ev.empty()) return 0;
    int rc = check_cuda(cudaEventSynchronize(g_prof.ev.back()), "prof sync");
    if (rc != AG_OK) return rc;
    g_prof.ms.assign(g_prof.ev.size(), 0.f);
    for (size_t i = 1; i < g_prof.ev.size(); i++) cudaEventElapsedTime(&g_prof.ms[i], g_prof.ev[i - 1], g_prof.ev[i]);
    return (int)g_prof.ev.size() - 1;
}

int ag_prof_get(int i, const char** name, float* ms) {
    AG_REQUIRE(i >= 0 && (size_t)(i + 1) < g_prof.ev.size() && name && ms, "index out of range");
    *name = g_prof.names[i + 1].c_str();
    *ms = g_prof.ms[i + 1];
    return AG_OK;
}

int ag_pyramid_plan(int B, int H, int W, int nlevels, double init_sigma, int border, ag_pyramid_plan_t* plan) {
    AG_REQUIRE(plan != nullptr, "plan is NULL");
    AG_REQUIRE(B >= 1 && H >= 1 && W >= 1, "bad image size");
    AG_REQUIRE(nlevels >= 1 && nlevels + 2 <= AG_MAX_LEVELS, "nlevels out of range");
    memset(plan, 0, sizeof(*plan));
    plan->B = B; plan->H = H; plan->W = W;
    plan->n_levels = nlevels + 2;
    // HandCraftedModules.py:15-22
    const double sigma_step = pow(2.0, 1.0 / (double)nlevels);
    const int min_size = 2 * border + 2 + 1;
    double cur_sigma = 0.5, first = 0.0, pd = 1.0;
    if (init_sigma > cur_sigma) {
        first = sqrt(init_sigma * init_sigma - cur_sigma * cur_sigma);
        cur_sigma = init_sigma;
    }
    int h = H, w = W, o = 0;
    long long off = 0;
    for (;;) {
        AG_REQUIRE(o < AG_MAX_OCTAVES, "too many octaves");
        plan->h[o] = h; plan->w[o] = w; plan->pix_dist[o] = pd;
        plan->sigma[o][0] = cur_sigma;
        plan->blur_sigma[o][0] = (o == 0) ? first : 0.0;
        for (int l = 0; l < plan->n_levels; l++) {
            plan->level_offset[o][l] = off;
            off += (long long)B * h * w;
        }
        for (int i = 1; i < plan->n_levels; i++) {  // HandCraftedModules.py:38-45
            plan->blur_sigma[o][i] = cur_sigma * sqrt(sigma_step * sigma_step - 1.0);
            cur_sigma = cur_sigma * sigma_step;
            plan->sigma[o][i] = cur_sigma;
        }
        o++;
        pd *= 2.0;
        cur_sigma = init_sigma;
        int nh = (h + 1) / 2, nw = (w + 1) / 2;
        if (nh <= min_size || nw <= min_size) break;  // HandCraftedModules.py:50
        h = nh; w = nw;
    }
    plan->n_octaves = o;
    plan->total_floats = off;
    return AG_OK;
}

int ag_gaussian_blur(const float* d_in, float* d_out, int B, int h, int w, double sigma, void* stream) {
    AG_REQUIRE(d_in && d_out && B >= 1 && h >= 1 && w >= 1, "bad arguments");
    return launch_blur(d_in, d_out, nullptr, B, h, w, sigma, (cudaStream_t)stream);
}

int ag_pyramid_build(const ag_pyramid_plan_t* p, const float* d_img, float* d_pyr, void* stream) {
    AG_REQUIRE(p && d_img && d_pyr, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int nl = p->n_levels, seed_level = nl - 2;  // level `nlevels` seeds the next octave (:46-47)
    // One launch per level: a one-launch-per-octave kernel was measured bit-identical but 2x slower (DESIGN.md section 5).
    for (int o = 0; o < p->n_octaves; o++) {
        const int h = p->h[o], w = p->w[o];
        float* lvl0 = d_pyr + p->level_offset[o][0];
        if (o == 0) {
            if (p->blur_sigma[0][0] > 0.0) {
                int rc = launch_blur(d_img, lvl0, nullptr, p->B, h, w, p->blur_sigma[0][0], st);
                if (rc != AG_OK) return rc;
            } else {
                int rc = check_cuda(cudaMemcpyAsync(lvl0, d_img, sizeof(float) * (size_t)p->B * h * w,
                                                    cudaMemcpyDeviceToDevice, st), "copy level 0");
                if (rc != AG_OK) return rc;
            }
        }
        for (int l = 1; l < nl; l++) {
            float* dec = (l == seed_level && o + 1 < p->n_octaves) ? d_pyr + p->level_offset[o + 1][0] : nullptr;
            int rc = launch_blur(d_pyr + p->level_offset[o][l - 1], d_pyr + p->level_offset[o][l], dec, p->B, h, w,
                                 p->blur_sigma[o][l], st);
            if (rc != AG_OK) return rc;
        }
    }
    return AG_OK;
}

}  // extern "C"
