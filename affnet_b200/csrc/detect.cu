// Hessian response, 3x3x3 NMS with sub-pixel soft-argmax, candidate compaction and global selection
// (SURVEY.md §8a rows a3-a6).
//
// Replaces HessianResp.forward (HandCraftedModules.py:58-78), NMS3d / NMS3dAndComposeA
// (HandCraftedModules.py:208-291) and the detection loop + global top-k of multiScaleDetector
// (SparseImgRepresenter.py:53-111).  Response maps never touch HBM in the fused path: each CTA stages a
// 36x36 window of three pyramid levels in shared memory, derives the three 34x34 response windows and
// runs NMS, border/octave-map masking, counting, soft-argmax and compaction from there.
//
// Integer exactness: given identical inputs the set of surviving pixels is identical to the reference's
// because every float op that decides survival is done in the reference's order with explicit
// non-contracted intrinsics (__fmul_rn/__fsub_rn/__fadd_rn): the Hessian determinant, `(x - max) + 1e-5 > 0`,
// `resp * (1 - octaveMap)` and the float->uint8 wrap of the octave map (Q4).
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace ag {

constexpr int DT = 32;            // output tile edge
constexpr int DNT = 256;          // threads per CTA
constexpr int RW = DT + 2;        // response window edge (tile + 1 halo)
constexpr int PW = DT + 4;        // pyramid window edge (tile + 2 halo)
constexpr int SEQ_PIX_BITS = 27;  // seq = slot << 27 | pixel

struct DetectOctave {
    const float* lvl[3];  // FROM_PYR: pyramid levels l-1,l,l+1 ([B,h,w]); else response maps low/cur/high
    float s4[3];          // sigma^4 (python double -> float32), FROM_PYR only
    float sc[3];          // scales as float32 (torch.FloatTensor(scales), Utils.py:133-135)
    int h, w, tiles_x, tiles_y, tile_base;
    int slot, prev_slot;  // level slot of this launch / of the previous detection level in the octave (-1: none)
    const uint8_t* P_in;  // resolved octave map before the previous level (NULL = zeros)
    const uint8_t* T_in;  // tentative map written by the previous level (valid iff that level had >1 positives)
    uint8_t* P_out;       // resolved map before THIS level (for the next level's fallback)
    uint8_t* T_out;       // tentative map after this level
};

struct DetectParams {
    DetectOctave oct[AG_MAX_OCTAVES];
    int n_oct, total_tiles;
    float th;
    int mr_border;
    int cand_cap, n_slots;
    float* cand_val;
    uint32_t* cand_seq;
    float* cand_scyx;
    int* cand_count;
    int* level_pos;
    int* level_emit;
};

__device__ __forceinline__ float hessian_at(const float (*s)[PW + 1], int py, int px, float s4, float th) {
    // (py,px) indexes the pyramid window; neighbours already hold replicate-clamped values.
    const float c = s[py][px];
    const float gxx = __fadd_rn(__fsub_rn(s[py][px - 1], __fmul_rn(2.0f, c)), s[py][px + 1]);
    const float gyy = __fadd_rn(__fsub_rn(s[py - 1][px], __fmul_rn(2.0f, c)), s[py + 1][px]);
    const float gxa = __fsub_rn(__fmul_rn(0.5f, s[py - 1][px - 1]), __fmul_rn(0.5f, s[py - 1][px + 1]));
    const float gxb = __fsub_rn(__fmul_rn(0.5f, s[py + 1][px - 1]), __fmul_rn(0.5f, s[py + 1][px + 1]));
    const float gxy = __fsub_rn(__fmul_rn(0.5f, gxa), __fmul_rn(0.5f, gxb));
    const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));
    const float r = __fmul_rn(fabsf(det), s4);
    return fmaxf(__fsub_rn(r, th), 0.0f);  // torch.clamp(resp - th, min=0), SparseImgRepresenter.py:77
}

__device__ __forceinline__ uint8_t float_to_u8_wrap(float v) {
    // torch-CPU float32 -> uint8: truncate toward zero, keep the low 8 bits (Q4).
    if (!(fabsf(v) < 2147483648.0f)) return 0;
    return (uint8_t)(__float2int_rz(v) & 0xFF);
}

template <bool FROM_PYR>
__global__ void __launch_bounds__(DNT) detect_level_kernel(const DetectParams P) {
    __shared__ float s_pyr[FROM_PYR ? 3 : 1][PW][PW + 1];
    __shared__ float s_resp[3][RW][RW + 1];
    __shared__ int s_cnt[3];  // pos, emit, base

    // locate octave for this tile
    int t = blockIdx.x, oi = 0;
#pragma unroll 1
    for (int i = 1; i < P.n_oct; i++)
        if (t >= P.oct[i].tile_base) oi = i;
    const DetectOctave& O = P.oct[oi];
    t -= O.tile_base;
    const int b = blockIdx.y;
    const int h = O.h, w = O.w;
    const int ty = t / O.tiles_x, tx = t - ty * O.tiles_x;
    const int y0 = ty * DT, x0 = tx * DT;
    const size_t img_off = (size_t)b * h * w;

    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;

    // ---- 1. response windows (origin y0-1, x0-1); zero outside the image (== conv zero padding) --------
    if (FROM_PYR) {
#pragma unroll
        for (int d = 0; d < 3; d++) {
            const float* src = O.lvl[d] + img_off;
            for (int i = threadIdx.x; i < PW * PW; i += DNT) {
                int ly = i / PW, lx = i - ly * PW;
                int gy = clampi(y0 - 2 + ly, 0, h - 1), gx = clampi(x0 - 2 + lx, 0, w - 1);
                s_pyr[FROM_PYR ? d : 0][ly][lx] = __ldg(src + (size_t)gy * w + gx);
            }
        }
        __syncthreads();
#pragma unroll
        for (int d = 0; d < 3; d++) {
            for (int i = threadIdx.x; i < RW * RW; i += DNT) {
                int ly = i / RW, lx = i - ly * RW;
                int gy = y0 - 1 + ly, gx = x0 - 1 + lx;
                float r = 0.f;
                if (gy >= 0 && gy < h && gx >= 0 && gx < w) r = hessian_at(s_pyr[FROM_PYR ? d : 0], ly + 1, lx + 1, O.s4[d], P.th);
                s_resp[d][ly][lx] = r;
            }
        }
    } else {
#pragma unroll
        for (int d = 0; d < 3; d++) {
            const float* src = O.lvl[d] + img_off;
            for (int i = threadIdx.x; i < RW * RW; i += DNT) {
                int ly = i / RW, lx = i - ly * RW;
                int gy = y0 - 1 + ly, gx = x0 - 1 + lx;
                s_resp[d][ly][lx] = (gy >= 0 && gy < h && gx >= 0 && gx < w) ? __ldg(src + (size_t)gy * w + gx) : 0.f;
            }
        }
    }
    __syncthreads();

    // ---- 2. per-pixel NMS + masking --------------------------------------------------------------------
    bool use_T = false;
    if (O.prev_slot >= 0 && O.T_in != nullptr) use_T = P.level_pos[b * P.n_slots + O.prev_slot] > 1;
    const uint8_t* om_src = use_T ? O.T_in : O.P_in;
    const bool border_ok = (P.mr_border < w) && (P.mr_border < h);  // Utils.py:141

    constexpr int PPT = DT * DT / DNT;  // 4 pixels per thread
    float vals[PPT];
    int n_pos = 0, n_emit = 0;
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        const int i = threadIdx.x + k * DNT;
        const int ly = i / DT, lx = i - ly * DT;
        const int gy = y0 + ly, gx = x0 + lx;
        float val = 0.f;
        if (gy < h && gx < w) {
            const float x = s_resp[1][ly + 1][lx + 1];
            float m = x;
#pragma unroll
            for (int d = 0; d < 3; d++)
#pragma unroll
                for (int dy = -1; dy <= 1; dy++)
#pragma unroll
                    for (int dx = -1; dx <= 1; dx++) {
                        const int ny = gy + dy, nx = gx + dx;
                        if (ny >= 0 && ny < h && nx >= 0 && nx < w) m = fmaxf(m, s_resp[d][ly + 1 + dy][lx + 1 + dx]);
                    }
            // NMS3d: ((x - m + eps) > 0) * x      HandCraftedModules.py:220
            float nms = (__fadd_rn(__fsub_rn(x, m), 1e-5f) > 0.f) ? x : 0.f;
            // zero_response_at_border(int(mrSize))   Utils.py:140-148
            if (!border_ok || gy < P.mr_border || gy >= h - P.mr_border || gx < P.mr_border || gx >= w - P.mr_border) nms = 0.f;
            const size_t p = img_off + (size_t)gy * w + gx;
            const uint8_t om = om_src ? om_src[p] : (uint8_t)0;
            val = __fmul_rn(nms, __fsub_rn(1.0f, (float)om));  // * (1 - octaveMap.float())   :246
            if (O.P_out) O.P_out[p] = om;
            if (O.T_out) O.T_out[p] = float_to_u8_wrap(__fadd_rn((float)om, val));  // (octaveMap.float()+resp).byte()  :256
            n_pos += (val > 0.f);
            n_emit += (val != 0.f);
        }
        vals[k] = val;
    }

    // ---- 3. counts and slot allocation -------------------------------------------------------------------
    const unsigned lane = threadIdx.x & 31;
    int wp = n_pos, we = n_emit;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        wp += __shfl_xor_sync(0xffffffffu, wp, o);
        we += __shfl_xor_sync(0xffffffffu, we, o);
    }
    // exclusive prefix of n_emit within the warp
    int incl = n_emit;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += v;
    }
    int warp_base = 0;
    if (lane == 0 && we > 0) {
        atomicAdd(&s_cnt[0], wp);
        warp_base = atomicAdd(&s_cnt[1], we);
    }
    warp_base = __shfl_sync(0xffffffffu, warp_base, 0);
    __syncthreads();
    if (threadIdx.x == 0 && s_cnt[1] > 0) {
        atomicAdd(&P.level_pos[b * P.n_slots + O.slot], s_cnt[0]);
        atomicAdd(&P.level_emit[b * P.n_slots + O.slot], s_cnt[1]);
        s_cnt[2] = atomicAdd(&P.cand_count[b], s_cnt[1]);
    }
    __syncthreads();
    if (n_emit == 0) return;
    int dst = s_cnt[2] + warp_base + (incl - n_emit);

    // ---- 4. soft-argmax + emission   HandCraftedModules.py:266-290 ------------------------------------
    const float min_size = (float)min(h, w);
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        if (vals[k] == 0.f) continue;
        const int i = threadIdx.x + k * DNT;
        const int ly = i / DT, lx = i - ly * DT;
        const int gy = y0 + ly, gx = x0 + lx;
        if (dst < P.cand_cap) {
            float ns = 0.f, ny = 0.f, nx = 0.f, den = 0.f;
#pragma unroll
            for (int d = 0; d < 3; d++)
#pragma unroll
                for (int dy = 0; dy < 3; dy++)
#pragma unroll
                    for (int dx = 0; dx < 3; dx++) {
                        const float r = s_resp[d][ly + dy][lx + dx];
                        ns = fmaf(O.sc[d], r, ns);
                        ny = fmaf(-0.5f + (float)dy, r, ny);  // offsets [-0.5, 0.5, 1.5]  (Q2)
                        nx = fmaf(-0.5f + (float)dx, r, nx);
                        den += r;
                    }
            den = __fadd_rn(den, 1e-8f);
            const float sc = __fdiv_rn(__fdiv_rn(ns, den), min_size);
            const float yy = __fdiv_rn(__fadd_rn(__fdiv_rn(ny, den), (float)gy), (float)h);
            const float xx = __fdiv_rn(__fadd_rn(__fdiv_rn(nx, den), (float)gx), (float)w);
            const size_t o = (size_t)b * P.cand_cap + dst;
            P.cand_val[o] = vals[k];
            P.cand_seq[o] = ((uint32_t)O.slot << SEQ_PIX_BITS) | (uint32_t)(gy * w + gx);
            P.cand_scyx[o * 3 + 0] = sc;
            P.cand_scyx[o * 3 + 1] = yy;
            P.cand_scyx[o * 3 + 2] = xx;
        }
        dst++;
    }
}


// ======================================================================================================================
// Single-launch detector for nlevels = 3 (the reference's only configuration): each pass reads all FIVE pyramid levels of its
// octave, derives the five response maps once, and runs the three detection levels together.  The reference's sequential
// octave-map logic (level k sees the map left by the accepted levels below it; a level with <= 1 positive maxima is dropped and
// leaves no trace, HandCraftedModules.py:246-256) is made launch-free by counting every acceptance hypothesis (a1, a2 in {0,1}) in
// the same pass and storing, with each candidate, the raw NMS values of the same pixel at the levels below; `resolve_kernel` then
// picks the branch the counters select and computes the masked response with the reference's exact fp32 / uint8-wrap arithmetic.
// ======================================================================================================================
constexpr int NVAR = 16;  // per (image, octave): [0] pos1, [1..2] pos2[a1], [3..6] pos3[a1][a2], [7] emit1, [8..9] emit2[a1], [10..13] emit3[a1][a2]

__device__ __forceinline__ uint8_t om_after(uint8_t om, float val) { return float_to_u8_wrap(__fadd_rn((float)om, val)); }
__device__ __forceinline__ float masked(float nms, uint8_t om) { return __fmul_rn(nms, __fsub_rn(1.0f, (float)om)); }


// ======================================================================================================================
// Register-resident formulation of the single-launch detector: one warp owns a band of rows of a 30-column strip (32 lanes = 30
// output columns + one response-halo column each side), walks down the rows keeping three pyramid rows of all five levels
// in registers, takes horizontal neighbours by warp shuffle, and never touches shared memory on the common path:
//   per pixel and level: 1 coalesced load + 2 shuffles + the Hessian; separable 3x3 max via 2 shuffles + FMNMX3.
// Candidates (about 1 % of the pixels) take a warp-cooperative slow path that gathers the 3x3x3 response neighbourhood by
// shuffle for the soft-argmax.
// ======================================================================================================================
constexpr int WCOLS = 30;   // output columns per warp strip
#ifndef AG_WROWS
#define AG_WROWS 48   // 32: 0.43 ms, 48: 0.40, 64: 0.39 per step of 16 images (4 halo rows per band); 48 keeps enough warps for one image
#endif
constexpr int WROWS = AG_WROWS;   // output rows per warp band
constexpr int WNT = 128;    // 4 warps per CTA, one band each

struct WarpOctave {
    const float* lvl[5];
    float s4[5], sc[5];
    int h, w, strips_x, bands_y, unit_base;   // unit = (band, strip)
};
struct WarpParams {
    WarpOctave oct[AG_MAX_OCTAVES];
    int n_oct, total_units;
    float th;
    int mr_border, cand_cap;
    float* cand_val;
    float* cand_aux;
    uint32_t* cand_seq;
    float* cand_scyx;
    int* cand_count;
    int* variants;
};

__device__ __forceinline__ float hessian_regs(float tl, float tc, float tr, float ml, float mc, float mr, float bl, float bc, float br, float s4, float th) {
    const float gxx = __fadd_rn(__fsub_rn(ml, __fmul_rn(2.0f, mc)), mr);
    const float gyy = __fadd_rn(__fsub_rn(tc, __fmul_rn(2.0f, mc)), bc);
    const float gxa = __fsub_rn(__fmul_rn(0.5f, tl), __fmul_rn(0.5f, tr));
    const float gxb = __fsub_rn(__fmul_rn(0.5f, bl), __fmul_rn(0.5f, br));
    const float gxy = __fsub_rn(__fmul_rn(0.5f, gxa), __fmul_rn(0.5f, gxb));
    const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));
    return fmaxf(__fsub_rn(__fmul_rn(fabsf(det), s4), th), 0.0f);
}

constexpr int WRING = 8;   // ring of pyramid rows per warp (cp.async prefetch distance WPD, 3 rows live)
constexpr int WPD = 5;
constexpr int WROWLEN = 34;  // 32 lane columns + one extra column each side
constexpr int WCBUF = 96;    // staged candidates per warp (a row yields at most 90); flushed with ONE atomic

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

template <int S0, int S1, int S2>   // response slots holding rows y-1, y, y+1
struct Slots {};

__global__ void __launch_bounds__(WNT) detect_warp_kernel(const WarpParams P) {
    __shared__ float s_ring[WNT / 32][WRING][5][WROWLEN];
    __shared__ float s_cbuf[WNT / 32][7][WCBUF];   // per-warp candidate staging: val, aux0, aux1, seq, sc, y, x
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int u = blockIdx.x * (WNT / 32) + wib;
    if (u >= P.total_units) return;
    int oi = 0;
#pragma unroll 1
    for (int i = 1; i < P.n_oct; i++)
        if (u >= P.oct[i].unit_base) oi = i;
    const WarpOctave& O = P.oct[oi];
    u -= O.unit_base;
    const int b = blockIdx.y, h = O.h, w = O.w;
    const int band = u / O.strips_x, strip = u - band * O.strips_x;
    const int r0 = band * WROWS;
    const int gx = strip * WCOLS - 1 + lane;            // lane's column; lanes 0 / 31 are the response halo
    const bool col_in = gx >= 0 && gx < w;
    const int cx = clampi(gx, 0, w - 1), cxl = clampi(gx - 1, 0, w - 1), cxr = clampi(gx + 1, 0, w - 1);
    const size_t img_off = (size_t)b * h * w;
    const bool border_ok = (P.mr_border < w) && (P.mr_border < h);
    const bool col_ok = lane >= 1 && lane <= WCOLS && col_in && border_ok && gx >= P.mr_border && gx < w - P.mr_border;
    const int rows_out = min(WROWS, h - r0);
    const int n_rows = rows_out + 4;                     // pyramid rows r0-2 .. r0+rows_out+1
    float (*ring)[5][WROWLEN] = s_ring[wib];

    auto issue_row = [&](int c) {                        // pyramid row r0-2+c -> ring slot c % WRING (replicate-clamped)
        if (c < n_rows) {
            const int cy = clampi(r0 - 2 + c, 0, h - 1);
#pragma unroll
            for (int d = 0; d < 5; d++) {
                const float* rowp = O.lvl[d] + img_off + (size_t)cy * w;
                float* dst = ring[c % WRING][d];
                cp_async4(dst + lane + 1, rowp + cx);
                if (lane == 0) cp_async4(dst, rowp + cxl);
                if (lane == 31) cp_async4(dst + 33, rowp + cxr);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    // rotating register state of the three most recent response rows (slot 0 = oldest): response, horizontal 3-max, and the
    // horizontal sums the soft-argmax needs (sum r, sum x_off * r), all taken from the same two shuffles
    float rs[5][3], rmx[5][3], hs[5][3], hx[5][3];
#pragma unroll
    for (int d = 0; d < 5; d++)
#pragma unroll
        for (int q = 0; q < 3; q++) { rs[d][q] = 0.f; rmx[d][q] = 0.f; hs[d][q] = 0.f; hx[d][q] = 0.f; }
    int var[14];
#pragma unroll
    for (int i = 0; i < 14; i++) var[i] = 0;
    const float min_size = (float)min(h, w);

    int buf_n = 0;   // warp-uniform
    float (*cbuf)[WCBUF] = s_cbuf[wib];
    auto flush = [&]() {
        if (buf_n == 0) return;
        int base = 0;
        if (lane == 0) base = atomicAdd(&P.cand_count[b], buf_n);
        base = __shfl_sync(0xffffffffu, base, 0);
        __syncwarp();
        for (int i = lane; i < buf_n; i += 32) {
            const int dst = base + i;
            if (dst < P.cand_cap) {
                const size_t o = (size_t)b * P.cand_cap + dst;
                P.cand_val[o] = cbuf[0][i];
                P.cand_aux[o * 2 + 0] = cbuf[1][i];
                P.cand_aux[o * 2 + 1] = cbuf[2][i];
                P.cand_seq[o] = __float_as_uint(cbuf[3][i]);
                P.cand_scyx[o * 3 + 0] = cbuf[4][i];
                P.cand_scyx[o * 3 + 1] = cbuf[5][i];
                P.cand_scyx[o * 3 + 2] = cbuf[6][i];
            }
        }
        __syncwarp();
        buf_n = 0;
    };

#pragma unroll 1
    for (int c = 0; c < WPD; c++) issue_row(c);
    // consume pyramid row c: response row (image row r0-3+c) enters slot 2; output row y = r0+c-4 sits in slot 1
#pragma unroll 1
    for (int c = 0; c < n_rows; c++) {
        asm volatile("cp.async.wait_group %0;" ::"n"(WPD - 1) : "memory");
        __syncwarp();
        if (c >= 2) {
            const int yy = r0 - 3 + c;
            const bool in = col_in && yy >= 0 && yy < h;
            const float (*t)[WROWLEN] = ring[(c - 2) % WRING];
            const float (*m)[WROWLEN] = ring[(c - 1) % WRING];
            const float (*bt)[WROWLEN] = ring[c % WRING];
#pragma unroll
            for (int d = 0; d < 5; d++) {
                rs[d][0] = rs[d][1]; rs[d][1] = rs[d][2]; rmx[d][0] = rmx[d][1]; rmx[d][1] = rmx[d][2];
                hs[d][0] = hs[d][1]; hs[d][1] = hs[d][2]; hx[d][0] = hx[d][1]; hx[d][1] = hx[d][2];
                float r = 0.f;
                if (in) r = hessian_regs(t[d][lane], t[d][lane + 1], t[d][lane + 2], m[d][lane], m[d][lane + 1], m[d][lane + 2], bt[d][lane], bt[d][lane + 1],
                                         bt[d][lane + 2], O.s4[d], P.th);
                float l = __shfl_up_sync(0xffffffffu, r, 1), rr = __shfl_down_sync(0xffffffffu, r, 1);
                if (lane == 0) l = 0.f;
                if (lane == 31) rr = 0.f;
                rs[d][2] = r;
                rmx[d][2] = fmaxf(fmaxf(l, r), rr);
                hs[d][2] = (l + r) + rr;
                hx[d][2] = fmaf(1.5f, rr, fmaf(0.5f, r, -0.5f * l));   // x offsets [-0.5, 0.5, 1.5] (Q2)
            }
        }
        if (c >= 4) {
            const int y = r0 + c - 4;
            float n1 = 0.f, n2 = 0.f, n3 = 0.f;
            if (col_ok && y >= P.mr_border && y < h - P.mr_border) {
                float M[5];
#pragma unroll
                for (int d = 0; d < 5; d++) M[d] = fmaxf(fmaxf(rmx[d][0], rmx[d][1]), rmx[d][2]);
                const float x1 = rs[1][1], x2 = rs[2][1], x3 = rs[3][1];
                n1 = (__fadd_rn(__fsub_rn(x1, fmaxf(fmaxf(M[0], M[1]), M[2])), 1e-5f) > 0.f) ? x1 : 0.f;   // NMS3d, HandCraftedModules.py:220
                n2 = (__fadd_rn(__fsub_rn(x2, fmaxf(fmaxf(M[1], M[2]), M[3])), 1e-5f) > 0.f) ? x2 : 0.f;
                n3 = (__fadd_rn(__fsub_rn(x3, fmaxf(fmaxf(M[2], M[3]), M[4])), 1e-5f) > 0.f) ? x3 : 0.f;
            }
            const unsigned m1 = __ballot_sync(0xffffffffu, n1 != 0.f), m2 = __ballot_sync(0xffffffffu, n2 != 0.f), m3 = __ballot_sync(0xffffffffu, n3 != 0.f);
            if (m1 | m2 | m3) {
                const int row_total = __popc(m1) + __popc(m2) + __popc(m3);
                if (buf_n + row_total > WCBUF) flush();
                if ((n1 != 0.f) || (n2 != 0.f) || (n3 != 0.f)) {
                    var[0] += n1 > 0.f; var[7] += n1 != 0.f;
#pragma unroll
                    for (int a1 = 0; a1 < 2; a1++) {
                        const uint8_t om1 = a1 ? om_after(0, n1) : (uint8_t)0;
                        const float v2 = masked(n2, om1);
                        var[1 + a1] += v2 > 0.f; var[8 + a1] += v2 != 0.f;
#pragma unroll
                        for (int a2 = 0; a2 < 2; a2++) {
                            const uint8_t om2 = a2 ? om_after(om1, v2) : om1;
                            const float v3 = masked(n3, om2);
                            var[3 + a1 * 2 + a2] += v3 > 0.f; var[10 + a1 * 2 + a2] += v3 != 0.f;
                        }
                    }
                    // soft-argmax (HandCraftedModules.py:266-290) from the rotating horizontal sums: no shuffles, no loop over lanes
                    const unsigned lt = (1u << lane) - 1u;
                    const float nn[3] = {n1, n2, n3};
                    const int pos[3] = {buf_n + __popc(m1 & lt), buf_n + __popc(m1) + __popc(m2 & lt), buf_n + __popc(m1) + __popc(m2) + __popc(m3 & lt)};
#pragma unroll
                    for (int q = 0; q < 3; q++) {
                        if (nn[q] == 0.f) continue;
                        float ns = 0.f, ny = 0.f, nx = 0.f, den = 0.f;
#pragma unroll
                        for (int d = 0; d < 3; d++) {
                            const float S = (hs[q + d][0] + hs[q + d][1]) + hs[q + d][2];
                            ns = fmaf(O.sc[q + d], S, ns);
                            ny += fmaf(1.5f, hs[q + d][2], fmaf(0.5f, hs[q + d][1], -0.5f * hs[q + d][0]));
                            nx += (hx[q + d][0] + hx[q + d][1]) + hx[q + d][2];
                            den += S;
                        }
                        den = __fadd_rn(den, 1e-8f);
                        const int dst = pos[q];
                        cbuf[0][dst] = nn[q];
                        cbuf[1][dst] = n1;
                        cbuf[2][dst] = n2;
                        cbuf[3][dst] = __uint_as_float(((uint32_t)(oi * 3 + q) << SEQ_PIX_BITS) | (uint32_t)(y * w + gx));
                        cbuf[4][dst] = __fdiv_rn(__fdiv_rn(ns, den), min_size);
                        cbuf[5][dst] = __fdiv_rn(__fadd_rn(__fdiv_rn(ny, den), (float)y), (float)h);
                        cbuf[6][dst] = __fdiv_rn(__fadd_rn(__fdiv_rn(nx, den), (float)gx), (float)w);
                    }
                }
                buf_n += row_total;
            }
        }
        __syncwarp();            // every lane has finished reading ring rows <= c before slot (c+WPD)%WRING is refilled
        issue_row(c + WPD);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    flush();
#pragma unroll
    for (int i = 0; i < 14; i++) {
        int v = var[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&P.variants[((size_t)b * P.n_oct + oi) * NVAR + i], v);
    }
}

// ======================================================================================================================
// Same detector, rows in registers (r02; ncu source view of detect_warp_kernel: 691 warp instructions per row, of which 155 issue the
// next row's cp.async through divergent halo branches and dynamically indexed constant loads, 45 re-read the 3x3 pyramid windows from
// shared memory, 40 rotate state registers, ~90 are the lone-lane soft-argmax divisions):
//   * every pyramid row is read from the ring ONCE (3 LDS per level); what later rows need of it stays in registers: the centre, the
//     half difference 0.5 l - 0.5 r (the gxy term of the rows above / below) and (l - 2 c) + r (gxx of the row itself) - the same
//     float operations in the same order as hessian_regs, so the response is bit-identical;
//   * the row loop is unrolled by three with compile-time slot indices: no register rotation;
//   * the row fetch is branch-free: one cp.async per level from a per-lane offset, the two halo columns by a predicated second one;
//   * the soft-argmax divisions move to the candidate flush, where 32 lanes finish 32 candidates at once.
// Records, counters and their semantics are those of detect_warp_kernel.
// ======================================================================================================================
template <int I> struct IC { static constexpr int value = I; };

template <int OFF>
__device__ __forceinline__ void cp_async4_off(uint32_t dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0 + %2], [%1], 4;" ::"r"(dst), "l"(src), "n"(OFF) : "memory");
}
template <int OFF>
__device__ __forceinline__ void cp_async4_off_if(uint32_t dst, const float* src, bool p) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %3, 0;\n @q cp.async.ca.shared.global [%0 + %2], [%1], 4;\n}\n" ::"r"(dst), "l"(src), "n"(OFF), "r"((uint32_t)p)
                 : "memory");
}

static_assert(WROWS <= 255, "8-bit per-lane hypothesis counters");
constexpr int RCB = 10;   // staged candidate record: val, n1, n2, seq, ns, ny, nx, den, y, x

#ifndef AG_DETROWS_MINB
#define AG_DETROWS_MINB 3   // 168 registers (4 B of spills), three CTAs per SM: 0.43 - 0.44 ms; 2 CTAs at 202 registers 0.47 - 0.49; 4 CTAs at 128 registers 0.59
#endif
__global__ void __launch_bounds__(WNT, AG_DETROWS_MINB) detect_rows_kernel(const WarpParams P) {
    __shared__ float s_ring[WNT / 32][WRING][5][WROWLEN];
    __shared__ float s_cbuf[WNT / 32][RCB][WCBUF];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int u = blockIdx.x * (WNT / 32) + wib;
    if (u >= P.total_units) return;
    int oi = 0;
#pragma unroll 1
    for (int i = 1; i < P.n_oct; i++)
        if (u >= P.oct[i].unit_base) oi = i;
    u -= P.oct[oi].unit_base;
    // octave constants into registers (dynamically indexed kernel parameters are constant-bank loads at every use otherwise)
    // (the five level pointers become one pointer + 32-bit element offsets: the levels of an octave lie in one pyramid allocation)
    const float* const lvl0 = P.oct[oi].lvl[0];
    int loff[5];
    float s4[5];
#pragma unroll
    for (int d = 0; d < 5; d++) { loff[d] = (int)(P.oct[oi].lvl[d] - lvl0); s4[d] = P.oct[oi].s4[d]; }
    const int h = P.oct[oi].h, w = P.oct[oi].w, strips_x = P.oct[oi].strips_x;
    const float th = P.th;
    const int b = blockIdx.y;
    const int band = u / strips_x, strip = u - band * strips_x;
    const int r0 = band * WROWS;
    const int gx = strip * WCOLS - 1 + lane;            // lane's column; lanes 0 / 31 are the response halo
    const bool col_in = gx >= 0 && gx < w;
    const int cx = clampi(gx, 0, w - 1);
    const bool halo_lane = lane == 0 || lane == 31;
    const int hdelta = (lane == 0 ? clampi(gx - 1, 0, w - 1) : clampi(gx + 1, 0, w - 1)) - cx;   // extra column of the halo lanes
    const int base_off = b * h * w + cx;                 // element offsets inside one pyramid allocation fit an int (ag_detect checks)
    const bool border_ok = (P.mr_border < w) && (P.mr_border < h);
    const bool col_ok = lane >= 1 && lane <= WCOLS && col_in && border_ok && gx >= P.mr_border && gx < w - P.mr_border;
    const int rows_out = min(WROWS, h - r0);
    const int n_rows = rows_out + 4;                     // pyramid rows r0-2 .. r0+rows_out+1
    float (*ring)[5][WROWLEN] = s_ring[wib];
    const uint32_t sdst = (uint32_t)__cvta_generic_to_shared(&ring[0][0][lane + 1]);
    const uint32_t sdst_h = (lane == 0) ? sdst - 4u : sdst + 4u;   // halo lanes: column 0 / 33

    auto issue_row = [&](int c) {                        // pyramid row r0-2+c -> ring slot c % WRING (replicate-clamped)
        if (c < n_rows) {
            const int cy = clampi(r0 - 2 + c, 0, h - 1);
            const int off = base_off + cy * w;
            const uint32_t so = (uint32_t)((c % WRING) * (5 * WROWLEN * 4));
            cp_async4_off<0 * WROWLEN * 4>(sdst + so, lvl0 + (loff[0] + off)); cp_async4_off_if<0 * WROWLEN * 4>(sdst_h + so, lvl0 + (loff[0] + off + hdelta), halo_lane);
            cp_async4_off<1 * WROWLEN * 4>(sdst + so, lvl0 + (loff[1] + off)); cp_async4_off_if<1 * WROWLEN * 4>(sdst_h + so, lvl0 + (loff[1] + off + hdelta), halo_lane);
            cp_async4_off<2 * WROWLEN * 4>(sdst + so, lvl0 + (loff[2] + off)); cp_async4_off_if<2 * WROWLEN * 4>(sdst_h + so, lvl0 + (loff[2] + off + hdelta), halo_lane);
            cp_async4_off<3 * WROWLEN * 4>(sdst + so, lvl0 + (loff[3] + off)); cp_async4_off_if<3 * WROWLEN * 4>(sdst_h + so, lvl0 + (loff[3] + off + hdelta), halo_lane);
            cp_async4_off<4 * WROWLEN * 4>(sdst + so, lvl0 + (loff[4] + off)); cp_async4_off_if<4 * WROWLEN * 4>(sdst_h + so, lvl0 + (loff[4] + off + hdelta), halo_lane);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    // per level and slot (slot = row index mod 3): pyramid-row terms pc (centre), ph (0.5 l - 0.5 r), pg ((l - 2 c) + r), and of the
    // response rows: response, horizontal 3-max, horizontal sums for the soft-argmax (sum r, sum x_off * r)
    float pc[5][3], ph[5][3], pg[5][3], rs[5][3], rmx[5][3], hs[5][3], hx[5][3];
#pragma unroll
    for (int d = 0; d < 5; d++)
#pragma unroll
        for (int q = 0; q < 3; q++) { pc[d][q] = 0.f; ph[d][q] = 0.f; pg[d][q] = 0.f; rs[d][q] = 0.f; rmx[d][q] = 0.f; hs[d][q] = 0.f; hx[d][q] = 0.f; }
    // hypothesis counters of this lane, four 8-bit counters per register (a lane counts at most once per row and counter: <= WROWS = 32)
    unsigned varp[4] = {0u, 0u, 0u, 0u};
    auto bump = [&](int i, bool cond) { varp[i >> 2] += cond ? (1u << ((i & 3) * 8)) : 0u; };
    const float min_size = (float)min(h, w);
    const float fh = (float)h, fw = (float)w;

    int buf_n = 0;   // warp-uniform
    float (*cbuf)[WCBUF] = s_cbuf[wib];
    auto flush = [&]() {
        if (buf_n == 0) return;
        int base = 0;
        if (lane == 0) base = atomicAdd(&P.cand_count[b], buf_n);
        base = __shfl_sync(0xffffffffu, base, 0);
        __syncwarp();
        for (int i = lane; i < buf_n; i += 32) {
            const int dst = base + i;
            if (dst < P.cand_cap) {
                const size_t o = (size_t)b * P.cand_cap + dst;
                const float ns = cbuf[4][i], ny = cbuf[5][i], nx = cbuf[6][i], den = cbuf[7][i];
                P.cand_val[o] = cbuf[0][i];
                P.cand_aux[o * 2 + 0] = cbuf[1][i];
                P.cand_aux[o * 2 + 1] = cbuf[2][i];
                P.cand_seq[o] = __float_as_uint(cbuf[3][i]);
                P.cand_scyx[o * 3 + 0] = __fdiv_rn(__fdiv_rn(ns, den), min_size);
                P.cand_scyx[o * 3 + 1] = __fdiv_rn(__fadd_rn(__fdiv_rn(ny, den), cbuf[8][i]), fh);
                P.cand_scyx[o * 3 + 2] = __fdiv_rn(__fadd_rn(__fdiv_rn(nx, den), cbuf[9][i]), fw);
            }
        }
        __syncwarp();
        buf_n = 0;
    };

    // consume pyramid row c (slot PN = c % 3): the response row of image row r0-3+c enters slot PN; output row y = r0+c-4 is the
    // response row of slot PM (one step old), its neighbours above / below are slots PO / PN
    auto step = [&](auto PC, const int c) {
        constexpr int PN = decltype(PC)::value, PM = (PN + 2) % 3, PO = (PN + 1) % 3;
        asm volatile("cp.async.wait_group %0;" ::"n"(WPD - 1) : "memory");
        __syncwarp();
        const float (*row)[WROWLEN] = ring[c % WRING];
        const int yy = r0 - 3 + c;
        const bool in = col_in && c >= 2 && yy >= 0 && yy < h;
#pragma unroll
        for (int d = 0; d < 5; d++) {
            const float L = row[d][lane], C = row[d][lane + 1], R = row[d][lane + 2];
            pc[d][PN] = C;
            ph[d][PN] = __fsub_rn(__fmul_rn(0.5f, L), __fmul_rn(0.5f, R));
            pg[d][PN] = __fadd_rn(__fsub_rn(L, __fmul_rn(2.0f, C)), R);
            // hessian_regs with t = slot PO, m = slot PM, b = this row
            const float gyy = __fadd_rn(__fsub_rn(pc[d][PO], __fmul_rn(2.0f, pc[d][PM])), C);
            const float gxy = __fsub_rn(__fmul_rn(0.5f, ph[d][PO]), __fmul_rn(0.5f, ph[d][PN]));
            const float det = __fsub_rn(__fmul_rn(pg[d][PM], gyy), __fmul_rn(gxy, gxy));
            float r = fmaxf(__fsub_rn(__fmul_rn(fabsf(det), s4[d]), th), 0.0f);
            r = in ? r : 0.f;
            float l = __shfl_up_sync(0xffffffffu, r, 1), rr = __shfl_down_sync(0xffffffffu, r, 1);
            l = (lane == 0) ? 0.f : l;
            rr = (lane == 31) ? 0.f : rr;
            rs[d][PN] = r;
            rmx[d][PN] = fmaxf(fmaxf(l, r), rr);
            hs[d][PN] = (l + r) + rr;
            hx[d][PN] = fmaf(1.5f, rr, fmaf(0.5f, r, -0.5f * l));   // x offsets [-0.5, 0.5, 1.5] (Q2)
        }
        if (c >= 4) {
            const int y = r0 + c - 4;
            float n1 = 0.f, n2 = 0.f, n3 = 0.f;
            if (col_ok && y >= P.mr_border && y < h - P.mr_border) {
                float M[5];
#pragma unroll
                for (int d = 0; d < 5; d++) M[d] = fmaxf(fmaxf(rmx[d][PO], rmx[d][PM]), rmx[d][PN]);
                const float x1 = rs[1][PM], x2 = rs[2][PM], x3 = rs[3][PM];
                n1 = (__fadd_rn(__fsub_rn(x1, fmaxf(fmaxf(M[0], M[1]), M[2])), 1e-5f) > 0.f) ? x1 : 0.f;   // NMS3d, HandCraftedModules.py:220
                n2 = (__fadd_rn(__fsub_rn(x2, fmaxf(fmaxf(M[1], M[2]), M[3])), 1e-5f) > 0.f) ? x2 : 0.f;
                n3 = (__fadd_rn(__fsub_rn(x3, fmaxf(fmaxf(M[2], M[3]), M[4])), 1e-5f) > 0.f) ? x3 : 0.f;
            }
            const unsigned m1 = __ballot_sync(0xffffffffu, n1 != 0.f), m2 = __ballot_sync(0xffffffffu, n2 != 0.f), m3 = __ballot_sync(0xffffffffu, n3 != 0.f);
            if (m1 | m2 | m3) {
                const int row_total = __popc(m1) + __popc(m2) + __popc(m3);
                if (buf_n + row_total > WCBUF) flush();
                if ((n1 != 0.f) || (n2 != 0.f) || (n3 != 0.f)) {
                    bump(0, n1 > 0.f); bump(7, n1 != 0.f);
#pragma unroll
                    for (int a1 = 0; a1 < 2; a1++) {
                        const uint8_t om1 = a1 ? om_after(0, n1) : (uint8_t)0;
                        const float v2 = masked(n2, om1);
                        bump(1 + a1, v2 > 0.f); bump(8 + a1, v2 != 0.f);
#pragma unroll
                        for (int a2 = 0; a2 < 2; a2++) {
                            const uint8_t om2 = a2 ? om_after(om1, v2) : om1;
                            const float v3 = masked(n3, om2);
                            bump(3 + a1 * 2 + a2, v3 > 0.f); bump(10 + a1 * 2 + a2, v3 != 0.f);
                        }
                    }
                    // soft-argmax sums (HandCraftedModules.py:266-290) from the horizontal sums of the three rows; the divisions wait for the flush
                    const unsigned lt = (1u << lane) - 1u;
                    const float nn[3] = {n1, n2, n3};
                    const int pos[3] = {buf_n + __popc(m1 & lt), buf_n + __popc(m1) + __popc(m2 & lt), buf_n + __popc(m1) + __popc(m2) + __popc(m3 & lt)};
#pragma unroll
                    for (int q = 0; q < 3; q++) {
                        if (nn[q] == 0.f) continue;
                        float ns = 0.f, ny = 0.f, nx = 0.f, den = 0.f;
#pragma unroll
                        for (int d = 0; d < 3; d++) {
                            const float S = (hs[q + d][PO] + hs[q + d][PM]) + hs[q + d][PN];
                            ns = fmaf(P.oct[oi].sc[q + d], S, ns);
                            ny += fmaf(1.5f, hs[q + d][PN], fmaf(0.5f, hs[q + d][PM], -0.5f * hs[q + d][PO]));
                            nx += (hx[q + d][PO] + hx[q + d][PM]) + hx[q + d][PN];
                            den += S;
                        }
                        const int dst = pos[q];
                        cbuf[0][dst] = nn[q];
                        cbuf[1][dst] = n1;
                        cbuf[2][dst] = n2;
                        cbuf[3][dst] = __uint_as_float(((uint32_t)(oi * 3 + q) << SEQ_PIX_BITS) | (uint32_t)(y * w + gx));
                        cbuf[4][dst] = ns;
                        cbuf[5][dst] = ny;
                        cbuf[6][dst] = nx;
                        cbuf[7][dst] = __fadd_rn(den, 1e-8f);
                        cbuf[8][dst] = (float)y;
                        cbuf[9][dst] = (float)gx;
                    }
                }
                buf_n += row_total;
            }
        }
        __syncwarp();            // every lane has read ring row c before slot (c+WPD) % WRING is refilled
        issue_row(c + WPD);
    };

#pragma unroll 1
    for (int c = 0; c < WPD; c++) issue_row(c);
#pragma unroll 1
    for (int c = 0; c < n_rows; c += 3) {
        step(IC<0>{}, c);
        if (c + 1 < n_rows) step(IC<1>{}, c + 1);
        if (c + 2 < n_rows) step(IC<2>{}, c + 2);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    flush();
#pragma unroll
    for (int i = 0; i < 14; i++) {
        int v = (int)((varp[i >> 2] >> ((i & 3) * 8)) & 0xFFu);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&P.variants[((size_t)b * P.n_oct + oi) * NVAR + i], v);
    }
}

// Picks the hypothesis branch the counters select, fills level_pos / level_emit, and turns every candidate's raw NMS value
// into the reference's masked response (or invalidates it: slot 31 is never accepted).
__global__ void resolve_kernel(const int* __restrict__ variants, int n_oct, int cand_cap, const int* __restrict__ cand_count,
                               float* __restrict__ cand_val, const float* __restrict__ cand_aux, uint32_t* __restrict__ cand_seq,
                               int* __restrict__ level_pos, int* __restrict__ level_emit) {
    __shared__ unsigned char s_a1[AG_MAX_OCTAVES], s_a2[AG_MAX_OCTAVES], s_a3[AG_MAX_OCTAVES];
    const int b = blockIdx.y;
    if (threadIdx.x < n_oct) {
        const int* v = variants + ((size_t)b * n_oct + threadIdx.x) * NVAR;
        const int a1 = v[0] > 1, a2 = v[1 + a1] > 1, a3 = v[3 + a1 * 2 + a2] > 1;
        s_a1[threadIdx.x] = a1; s_a2[threadIdx.x] = a2; s_a3[threadIdx.x] = a3;
        if (blockIdx.x == 0) {
            int* lp = level_pos + ((size_t)b * n_oct + threadIdx.x) * 3;
            int* le = level_emit + ((size_t)b * n_oct + threadIdx.x) * 3;
            lp[0] = v[0]; lp[1] = v[1 + a1]; lp[2] = v[3 + a1 * 2 + a2];
            le[0] = v[7]; le[1] = v[8 + a1]; le[2] = v[10 + a1 * 2 + a2];
        }
    }
    __syncthreads();
    const int n = min(cand_count[b], cand_cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const size_t o = (size_t)b * cand_cap + i;
        const uint32_t sq = cand_seq[o];
        const int slot = (int)(sq >> SEQ_PIX_BITS), oc = slot / 3, q = slot - oc * 3;
        const int a1 = s_a1[oc], a2 = s_a2[oc], a3 = s_a3[oc];
        const float n1 = cand_aux[o * 2], n2 = cand_aux[o * 2 + 1], raw = cand_val[o];
        const uint8_t om1 = a1 ? om_after(0, n1) : (uint8_t)0;
        float val;
        bool acc;
        if (q == 0) { val = raw; acc = a1; }
        else if (q == 1) { val = masked(raw, om1); acc = a2; }
        else {
            const float v2 = masked(n2, om1);
            const uint8_t om2 = a2 ? om_after(om1, v2) : om1;
            val = masked(raw, om2); acc = a3;
        }
        if (!acc || val == 0.f) cand_seq[o] = 0xFFFFFFFFu;
        else cand_val[o] = val;
    }
}

// ---- standalone Hessian response map (HessianResp module API + parity tests) -------------------------
__global__ void hessian_kernel(const float* __restrict__ in, float* __restrict__ out, int h, int w, float s4, float th) {
    __shared__ float s[PW][PW + 1];  // uses the (DT+2)^2 corner of the window
    const int b = blockIdx.z, y0 = blockIdx.y * DT, x0 = blockIdx.x * DT;
    const float* src = in + (size_t)b * h * w;
    for (int i = threadIdx.x; i < RW * RW; i += DNT) {
        int ly = i / RW, lx = i - ly * RW;
        int gy = clampi(y0 - 1 + ly, 0, h - 1), gx = clampi(x0 - 1 + lx, 0, w - 1);
        s[ly][lx] = __ldg(src + (size_t)gy * w + gx);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < DT * DT; i += DNT) {
        int ly = i / DT, lx = i - ly * DT;
        int gy = y0 + ly, gx = x0 + lx;
        if (gy < h && gx < w) out[(size_t)b * h * w + (size_t)gy * w + gx] = hessian_at(s, ly + 1, lx + 1, s4, th);
    }
}

// ---- global selection ---------------------------------------------------------------------------------
constexpr int SNT = 1024;

struct SelectParams {
    const float* cand_val;
    const uint32_t* cand_seq;
    const float* cand_scyx;
    const int* cand_count;
    const int* level_pos;
    const int* level_emit;
    int cand_cap, n_slots, n_det;  // n_det = detection levels per octave
    int num_features, out_cap, sort_cap;  // sort_cap: power of two >= max selectable
    float a_scale;
    float* resp;
    float* lafs;
    int* oct;
    int* lvl;
    int* count;
};

// A cluster of SEL_CL CTAs per image (thread-block cluster, distributed shared memory): every CTA scans 1/SEL_CL of the candidate list,
// the per-pass histograms of the radix select are merged by CTA 0 through DSMEM, the selected candidates are appended to CTA 0's sort
// buffer with DSMEM atomics, and CTA 0 sorts and writes the output.  The radix select stops as soon as the chosen digit's bucket is needed
// entirely (typically after 2-3 of the 8 passes).  (r01: one CTA per image, 8 full passes, serial histogram scan: 0.18 ms for 16 images,
// 0.88 ms for one 4K image.)
constexpr int SEL_CL = 8;

__device__ __forceinline__ uint32_t dsmem_addr(const void* p, int rank) {
    uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ int dsmem_ld_i32(uint32_t a) { int v; asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ unsigned long long dsmem_ld_u64(uint32_t a) { unsigned long long v; asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void dsmem_st_i32(uint32_t a, int v) { asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void dsmem_st_u64(uint32_t a, unsigned long long v) { asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ int dsmem_atomic_add(uint32_t a, int v) { int o; asm volatile("atom.shared::cluster.add.s32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__global__ void __launch_bounds__(SNT) select_kernel(const SelectParams P) {
    extern __shared__ unsigned char smem_raw[];
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(smem_raw);                                    // used by cluster rank 0
    int* s_idx = reinterpret_cast<int*>(smem_raw + sizeof(unsigned long long) * P.sort_cap);
    __shared__ int s_hist[256];
    __shared__ unsigned s_accept;  // bit per slot
    __shared__ int s_misc[4];      // 0: sorted mode, 1: m (number to select), 2: still needed inside the chosen digit / done flag (rank 0), 3: fill counter (rank 0)
    __shared__ unsigned long long s_prefix;   // rank 0 publishes the radix prefix here
    __shared__ int s_ctl[2];       // rank 0: [0] remaining, [1] done

    unsigned rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int b = blockIdx.x / SEL_CL;
    const int n = min(P.cand_count[b], P.cand_cap);
    const float* val = P.cand_val + (size_t)b * P.cand_cap;
    const uint32_t* seq = P.cand_seq + (size_t)b * P.cand_cap;
    const int nf = P.num_features;

    if (threadIdx.x == 0) {   // every CTA of the cluster derives the same selection parameters
        unsigned acc = 0;
        long long total = 0;
        bool trimmed = false;
        for (int s = 0; s < P.n_slots; s++) {
            const int pos = P.level_pos[b * P.n_slots + s], emit = P.level_emit[b * P.n_slots + s];
            if (pos > 1) {  // HandCraftedModules.py:253
                acc |= 1u << s;
                if (nf > 0 && nf < pos) { total += nf; trimmed = true; }  // per-level topk :259
                else total += emit;
            }
        }
        s_accept = acc;
        const bool sorted = (nf > 0) && (total > nf || trimmed);  // SparseImgRepresenter.py:104
        long long m = sorted ? nf : total;
        if (m > P.out_cap) m = P.out_cap;
        if (m > n) m = n;
        s_misc[0] = sorted;
        s_misc[1] = (int)m;
        s_misc[3] = 0;
        s_prefix = 0ull;
        s_ctl[0] = (int)m; s_ctl[1] = 0;
    }
    __syncthreads();
    const unsigned accept = s_accept;
    const bool sorted = s_misc[0] != 0;
    const int m = s_misc[1];

    auto key_of = [&](int i) -> unsigned long long {
        const uint32_t sq = seq[i];
        if (!((accept >> (sq >> SEQ_PIX_BITS)) & 1u)) return 0ull;
        const unsigned long long lo = (unsigned long long)(0xFFFFFFFFu - sq);
        // +1 keeps every valid key above the invalid key 0
        return sorted ? (((unsigned long long)float_to_ordered(val[i]) << 32) | lo) : (lo + 1ull);
    };
    const uint32_t r0_prefix = dsmem_addr(&s_prefix, 0), r0_ctl = dsmem_addr(s_ctl, 0);
    const uint32_t r0_fill = dsmem_addr(&s_misc[3], 0), r0_key = dsmem_addr(s_key, 0), r0_idx = dsmem_addr(s_idx, 0);

    unsigned long long kth = 1ull;   // unsorted mode: every valid key (>= 1) is taken
    if (m > 0 && sorted) {
        // radix select of the m-th largest key, 8 bits per pass from the top; candidates are dealt round-robin to the CTAs of the cluster
        unsigned long long prefix = 0ull;
        for (int pass = 7; pass >= 0; pass--) {
            for (int i = threadIdx.x; i < 256; i += SNT) s_hist[i] = 0;
            __syncthreads();
            const int shift = pass * 8;
            const unsigned long long hi_mask = (pass == 7) ? 0ull : (~0ull << (shift + 8));
            for (int i = (int)rank * SNT + threadIdx.x; i < n; i += SEL_CL * SNT) {
                const unsigned long long k = key_of(i);
                if ((k & hi_mask) == prefix) atomicAdd(&s_hist[(int)((k >> shift) & 0xFF)], 1);
            }
            cluster_sync_all();                      // all local histograms complete
            if (rank == 0) {
                if (threadIdx.x < 256) {             // merge the other CTAs' histograms into this one
                    int t = s_hist[threadIdx.x];
                    for (int r = 1; r < SEL_CL; r++) t += dsmem_ld_i32(dsmem_addr(&s_hist[threadIdx.x], r));
                    s_hist[threadIdx.x] = t;
                }
                __syncthreads();
                if (threadIdx.x < 32) {              // warp 0: suffix sums over the 256 bins, 8 bins per lane (lane 31 = top digits)
                    const int lane = threadIdx.x;
                    int loc[8], tot = 0;
#pragma unroll
                    for (int j = 0; j < 8; j++) { loc[j] = s_hist[lane * 8 + j]; tot += loc[j]; }
                    int above = tot;                 // inclusive suffix sum over lanes >= lane
                    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(0xffffffffu, above, o); if (lane + o < 32) above += t; }
                    above -= tot;                    // keys in strictly higher lanes
                    const int remaining = s_ctl[0];
                    // the digit d with  count(> d) < remaining <= count(>= d)
                    int cum = above, dsel = -1, need = 0, cnt = 0;
#pragma unroll
                    for (int j = 7; j >= 0; j--) {
                        if (dsel < 0 && cum < remaining && cum + loc[j] >= remaining) { dsel = lane * 8 + j; need = remaining - cum; cnt = loc[j]; }
                        cum += loc[j];
                    }
                    const unsigned hit = __ballot_sync(0xffffffffu, dsel >= 0);
                    if (hit == 0) { if (lane == 0) { s_ctl[1] = 1; } }        // fewer valid keys than requested (cannot happen: m <= n valid): stop
                    else if (lane == (int)(31 - __clz(hit))) {                  // the highest lane that found it
                        s_prefix = prefix | ((unsigned long long)dsel << shift);
                        s_ctl[0] = need;
                        s_ctl[1] = (need == cnt) ? 1 : 0;                       // the whole bucket is needed: its lower bits need no refinement
                    }
                }
            }
            cluster_sync_all();                      // rank 0 has published prefix / remaining / done
            prefix = dsmem_ld_u64(r0_prefix);        // (rank 0 rewrites them only after the next pass's first cluster barrier)
            const int done = dsmem_ld_i32(r0_ctl + 4);
            if (done) break;
        }
        kth = prefix;   // keys are unique (seq unique): exactly m keys are >= kth (lower bits zero when stopped early)
    }
    if (m > 0) {
        if (rank == 0) {
            for (int i = threadIdx.x; i < P.sort_cap; i += SNT) { s_key[i] = 0ull; s_idx[i] = -1; }
        }
        cluster_sync_all();
        for (int i = (int)rank * SNT + threadIdx.x; i < n; i += SEL_CL * SNT) {
            const unsigned long long k = key_of(i);
            if (k >= kth && k != 0ull) {
                const int pos = dsmem_atomic_add(r0_fill, 1);
                if (pos < P.sort_cap) { dsmem_st_u64(r0_key + (uint32_t)pos * 8u, k); dsmem_st_i32(r0_idx + (uint32_t)pos * 4u, i); }
            }
        }
    }
    cluster_sync_all();                              // the sort buffer of rank 0 is complete; the other CTAs are done
    if (rank != 0) return;
    if (m > 0) {
        if (threadIdx.x == 0 && s_misc[3] < s_misc[1]) s_misc[1] = s_misc[3];  // candidate list overflowed
        __syncthreads();
        bitonic_sort_desc<true>(s_key, s_idx, P.sort_cap);   // descending by key
    }
    // outputs
    __syncthreads();
    const int m_out = s_misc[1];
    const float* scyx = P.cand_scyx + (size_t)b * P.cand_cap * 3;
    for (int i = threadIdx.x; i < m_out; i += SNT) {
        const int c = s_idx[i];
        const size_t o = (size_t)b * P.out_cap + i;
        const float sc = __fmul_rn(P.a_scale, scyx[c * 3 + 0]);  // mrSize * LAFs[:, :, 0:2]   SparseImgRepresenter.py:198
        P.resp[o] = val[c];
        float* L = P.lafs + o * 6;
        L[0] = sc; L[1] = 0.f; L[2] = scyx[c * 3 + 2];
        L[3] = 0.f; L[4] = sc; L[5] = scyx[c * 3 + 1];
        const int slot = (int)(seq[c] >> SEQ_PIX_BITS);
        P.oct[o] = slot / P.n_det;
        P.lvl[o] = slot % P.n_det;  // detection level_idx - 1: patches come from the level below (:94)
    }
    // a candidate list that overflowed its capacity is reported as count = -1 (downstream kernels then process no rows)
    if (threadIdx.x == 0) P.count[b] = (P.cand_count[b] > P.cand_cap) ? -1 : m_out;
}

}  // namespace ag

using namespace ag;

extern "C" {

size_t ag_detect_ws_bytes(const ag_pyramid_plan_t* p, int cand_cap) {
    if (!p || cand_cap <= 0) return 0;
    const size_t B = p->B, slots = (size_t)p->n_octaves * (p->n_levels - 2);
    size_t n = 0;
    n += align_up(B * cand_cap * sizeof(float), 256);
    n += align_up(B * cand_cap * sizeof(uint32_t), 256);
    n += align_up(B * cand_cap * 3 * sizeof(float), 256);
    n += align_up(B * cand_cap * 2 * sizeof(float), 256);
    n += align_up((B + 2 * B * slots + B * (size_t)p->n_octaves * NVAR) * sizeof(int), 256);
    size_t px = 0;
    for (int o = 0; o < p->n_octaves; o++) px += (size_t)p->h[o] * p->w[o];
    n += align_up(4 * B * px, 256);
    return n;
}

int ag_detect_ws_carve(const ag_pyramid_plan_t* p, int cand_cap, void* d_ws, ag_detect_ws_t* ws) {
    AG_REQUIRE(p && d_ws && ws && cand_cap > 0, "bad arguments");
    const size_t B = p->B, slots = (size_t)p->n_octaves * (p->n_levels - 2);
    AG_REQUIRE(slots <= 32, "too many detection levels (max 32 slots)");
    AG_REQUIRE((long long)p->H * p->W < (1ll << SEQ_PIX_BITS), "image too large for the candidate key");
    unsigned char* c = (unsigned char*)d_ws;
    ws->B = p->B; ws->cand_cap = cand_cap; ws->n_level_slots = (int)slots;
    ws->d_cand_val = (float*)c; c += align_up(B * cand_cap * sizeof(float), 256);
    ws->d_cand_seq = (uint32_t*)c; c += align_up(B * cand_cap * sizeof(uint32_t), 256);
    ws->d_cand_scyx = (float*)c; c += align_up(B * cand_cap * 3 * sizeof(float), 256);
    ws->d_cand_aux = (float*)c; c += align_up(B * cand_cap * 2 * sizeof(float), 256);
    ws->d_cand_count = (int*)c;
    ws->d_level_pos = ws->d_cand_count + B;
    ws->d_level_emit = ws->d_level_pos + B * slots;
    ws->d_variants = ws->d_level_emit + B * slots;
    c += align_up((B + 2 * B * slots + B * (size_t)p->n_octaves * NVAR) * sizeof(int), 256);
    ws->d_octave_maps = c;
    return AG_OK;
}

static int fill_common(DetectParams& P, const ag_detect_ws_t* ws, float th, int mr_border) {
    P.th = th; P.mr_border = mr_border;
    P.cand_cap = ws->cand_cap; P.n_slots = ws->n_level_slots;
    P.cand_val = ws->d_cand_val; P.cand_seq = ws->d_cand_seq; P.cand_scyx = ws->d_cand_scyx;
    P.cand_count = ws->d_cand_count; P.level_pos = ws->d_level_pos; P.level_emit = ws->d_level_emit;
    return AG_OK;
}

int ag_detect(const ag_pyramid_plan_t* p, const float* d_pyr, float th, int mr_border, ag_detect_ws_t* ws, void* stream) {
    AG_REQUIRE(p && d_pyr && ws, "NULL argument");
    AG_REQUIRE(ws->B == p->B, "workspace batch mismatch");
    cudaStream_t st = (cudaStream_t)stream;
    const int n_det = p->n_levels - 2;
    AG_REQUIRE(ws->n_level_slots == p->n_octaves * n_det, "workspace slot mismatch");
    const size_t B = p->B;
    int rc = check_cuda(cudaMemsetAsync(ws->d_cand_count, 0, (B + 2 * B * ws->n_level_slots + B * (size_t)p->n_octaves * NVAR) * sizeof(int), st),
                        "memset counters");
    if (rc != AG_OK) return rc;
    if (n_det == 3) {
        // single-launch detector + hypothesis resolution
        WarpParams Wp;
        memset(&Wp, 0, sizeof(Wp));
        Wp.n_oct = p->n_octaves; Wp.th = th; Wp.mr_border = mr_border; Wp.cand_cap = ws->cand_cap;
        Wp.cand_val = ws->d_cand_val; Wp.cand_aux = ws->d_cand_aux; Wp.cand_seq = ws->d_cand_seq; Wp.cand_scyx = ws->d_cand_scyx;
        Wp.cand_count = ws->d_cand_count; Wp.variants = ws->d_variants;
        int units = 0;
        for (int o = 0; o < p->n_octaves; o++) {
            WarpOctave& O = Wp.oct[o];
            for (int d = 0; d < 5; d++) {
                O.lvl[d] = d_pyr + p->level_offset[o][d];
                O.s4[d] = (float)pow(p->sigma[o][d], 4.0);
                O.sc[d] = (float)p->sigma[o][d];
            }
            O.h = p->h[o]; O.w = p->w[o];
            O.strips_x = cdiv(O.w, WCOLS); O.bands_y = cdiv(O.h, WROWS);
            O.unit_base = units;
            units += O.strips_x * O.bands_y;
        }
        Wp.total_units = units;
        static const bool use_v1 = getenv("AG_DETECT_WARP_V1") != nullptr;     // A/B switch: the first register formulation
        // detect_rows_kernel addresses an octave's levels with 32-bit element offsets from its first level
        bool fits32 = true;
        for (int o = 0; o < p->n_octaves; o++) {
            long long lo = 0, hi = 0;
            for (int d = 0; d < 5; d++) { const long long off = Wp.oct[o].lvl[d] - Wp.oct[o].lvl[0]; lo = off < lo ? off : lo; hi = off > hi ? off : hi; }
            if (lo < -(1ll << 30) || hi + (long long)p->B * p->h[o] * p->w[o] >= (1ll << 31) - 64) fits32 = false;
        }
        if (use_v1 || !fits32) {
            detect_warp_kernel<<<dim3(cdiv(units, WNT / 32), p->B), WNT, 0, st>>>(Wp);
            AG_CHECK_LAUNCH("detect_warp_kernel");
        } else {
            detect_rows_kernel<<<dim3(cdiv(units, WNT / 32), p->B), WNT, 0, st>>>(Wp);
            AG_CHECK_LAUNCH("detect_rows_kernel");
        }
        resolve_kernel<<<dim3(8, p->B), 256, 0, st>>>(ws->d_variants, p->n_octaves, ws->cand_cap, ws->d_cand_count, ws->d_cand_val, ws->d_cand_aux,
                                                       ws->d_cand_seq, ws->d_level_pos, ws->d_level_emit);
        AG_CHECK_LAUNCH("resolve_kernel");
        return AG_OK;
    }
    // octave-map scratch: every octave owns 4 uint8 maps [B,h,w] (resolved P and tentative T, ping-ponged),
    // packed octave after octave: 4 * sum_o B*h_o*w_o bytes in total.
    for (int k = 0; k < n_det; k++) {
        DetectParams P;
        memset(&P, 0, sizeof(P));
        fill_common(P, ws, th, mr_border);
        P.n_oct = p->n_octaves;
        int tiles = 0;
        size_t oct_off = 0;
        for (int o = 0; o < p->n_octaves; o++) {
            DetectOctave& O = P.oct[o];
            const int l = k + 1;
            for (int d = 0; d < 3; d++) {
                O.lvl[d] = d_pyr + p->level_offset[o][l - 1 + d];
                const double s = p->sigma[o][l - 1 + d];
                O.s4[d] = (float)pow(s, 4.0);  // python `scale**4` (double pow), cast to float32 by torch's scalar mul
                O.sc[d] = (float)s;
            }
            O.h = p->h[o]; O.w = p->w[o];
            O.tiles_x = cdiv(O.w, DT); O.tiles_y = cdiv(O.h, DT);
            O.tile_base = tiles;
            tiles += O.tiles_x * O.tiles_y;
            O.slot = o * n_det + k;
            O.prev_slot = (k > 0) ? O.slot - 1 : -1;
            uint8_t* base = ws->d_octave_maps;
            const size_t osz = B * (size_t)O.h * O.w;
            uint8_t* r = base + 4 * oct_off;
            uint8_t* Pbuf[2] = {r, r + osz};
            uint8_t* Tbuf[2] = {r + 2 * osz, r + 3 * osz};
            O.P_in = (k >= 2) ? Pbuf[(k - 1) & 1] : nullptr;   // resolved map before level k-1 (zeros for k-1 == 0)
            O.T_in = (k >= 1) ? Tbuf[(k - 1) & 1] : nullptr;   // tentative map after level k-1
            O.P_out = (k >= 1 && k + 1 < n_det) ? Pbuf[k & 1] : nullptr;
            O.T_out = (k + 1 < n_det) ? Tbuf[k & 1] : nullptr;
            oct_off += osz;
        }
        P.total_tiles = tiles;
        dim3 grid(tiles, p->B);
        detect_level_kernel<true><<<grid, DNT, 0, st>>>(P);
        AG_CHECK_LAUNCH("detect_level_kernel");
    }
    return AG_OK;
}

int ag_detect_level_from_responses(const float* d_low, const float* d_cur, const float* d_high, int h, int w,
                                   const double scales[3], int mr_border, const uint8_t* d_omap_in, uint8_t* d_omap_out,
                                   int slot, ag_detect_ws_t* ws, void* stream) {
    AG_REQUIRE(d_low && d_cur && d_high && ws && scales, "NULL argument");
    AG_REQUIRE(ws->B == 1, "single-image entry point");
    AG_REQUIRE(slot >= 0 && slot < ws->n_level_slots, "slot out of range");
    DetectParams P;
    memset(&P, 0, sizeof(P));
    fill_common(P, ws, 0.f, mr_border);
    P.n_oct = 1;
    DetectOctave& O = P.oct[0];
    O.lvl[0] = d_low; O.lvl[1] = d_cur; O.lvl[2] = d_high;
    for (int d = 0; d < 3; d++) { O.sc[d] = (float)scales[d]; O.s4[d] = 1.f; }
    O.h = h; O.w = w; O.tiles_x = cdiv(w, DT); O.tiles_y = cdiv(h, DT); O.tile_base = 0;
    O.slot = slot; O.prev_slot = -1;
    O.P_in = d_omap_in; O.T_in = nullptr; O.P_out = nullptr; O.T_out = d_omap_out;
    P.total_tiles = O.tiles_x * O.tiles_y;
    detect_level_kernel<false><<<dim3(P.total_tiles, 1), DNT, 0, (cudaStream_t)stream>>>(P);
    AG_CHECK_LAUNCH("detect_level_kernel<resp>");
    return AG_OK;
}

int ag_hessian_response(const float* d_in, float* d_out, int B, int h, int w, double sigma, float th, void* stream) {
    AG_REQUIRE(d_in && d_out && B >= 1 && h >= 1 && w >= 1, "bad arguments");
    dim3 grid(cdiv(w, DT), cdiv(h, DT), B);
    hessian_kernel<<<grid, DNT, 0, (cudaStream_t)stream>>>(d_in, d_out, h, w, (float)pow(sigma, 4.0), th);
    AG_CHECK_LAUNCH("hessian_kernel");
    return AG_OK;
}

int ag_select_keypoints(const ag_pyramid_plan_t* p, const ag_detect_ws_t* ws, int num_features, float a_scale, int out_cap,
                        float* d_resp, float* d_lafs, int* d_oct, int* d_lvl, int* d_count, void* stream) {
    AG_REQUIRE(p && ws && d_resp && d_lafs && d_oct && d_lvl && d_count, "NULL argument");
    AG_REQUIRE(out_cap >= 1, "out_cap must be positive");
    const int need = (num_features > 0) ? (num_features < out_cap ? num_features : out_cap) : out_cap;
    int sort_cap = 32;
    while (sort_cap < need) sort_cap <<= 1;
    const size_t smem = (size_t)sort_cap * (sizeof(unsigned long long) + sizeof(int));
    if (smem > 200 * 1024) {
        set_error("ag_select_keypoints: selecting %d keypoints needs %zu B of shared memory (max 200 KiB)", need, smem);
        return AG_ERR_CAPACITY;
    }
    static size_t configured[64] = {};   // per device (ADVICE r01: the attribute is per device)
    int dev = 0;
    cudaGetDevice(&dev);
    if (smem > 32 * 1024 && smem > configured[dev & 63]) {  // static + dynamic must stay under the 48 KiB default
        int rc = check_cuda(cudaFuncSetAttribute(select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "select smem attr");
        if (rc != AG_OK) return rc;
        configured[dev & 63] = smem;
    }
    SelectParams S;
    S.cand_val = ws->d_cand_val; S.cand_seq = ws->d_cand_seq; S.cand_scyx = ws->d_cand_scyx;
    S.cand_count = ws->d_cand_count; S.level_pos = ws->d_level_pos; S.level_emit = ws->d_level_emit;
    S.cand_cap = ws->cand_cap; S.n_slots = ws->n_level_slots; S.n_det = p->n_levels - 2;
    S.num_features = num_features; S.out_cap = out_cap; S.sort_cap = sort_cap; S.a_scale = a_scale;
    S.resp = d_resp; S.lafs = d_lafs; S.oct = d_oct; S.lvl = d_lvl; S.count = d_count;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(ws->B * SEL_CL); cfg.blockDim = dim3(SNT); cfg.dynamicSmemBytes = smem; cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = SEL_CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int rcl = check_cuda(cudaLaunchKernelEx(&cfg, select_kernel, S), "select_kernel launch");
    if (rcl != AG_OK) return rcl;
    AG_CHECK_LAUNCH("select_kernel");
    return AG_OK;
}

}  // extern "C"
