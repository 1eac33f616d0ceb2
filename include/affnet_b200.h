/*
 * affnet_b200 C ABI  --  the drop-in boundary of the B200-native HesAffNet + HardNet hot path.
 *
 * The reference (ducha-aiki/affnet) has no FFI: its boundary is the Python module API
 * (SURVEY.md §8b).  The thin Python mirror in `affnet_b200/` keeps those names and calls ONLY the
 * entry points below (ctypes).  Each entry point cites the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every `d_*` pointer is DEVICE memory owned by the caller,
 *     every `h_*` pointer is HOST memory.  The library never allocates result buffers and never
 *     synchronises the stream (except the two `*_create` functions, which upload weights).
 *   - `stream` is a `cudaStream_t` passed as `void*`; all work is enqueued on it.
 *   - return value: 0 on success, negative `AG_ERR_*` otherwise; `ag_last_error()` gives a message.
 *   - images / pyramid levels are float32 `[B, h, w]` (single channel, batch-major), 0..255 scale.
 *   - LAFs are float32 `[n, 2, 3]` = [[a11 a12 x], [a21 a22 y]]; "normalised" means A in units of
 *     min(h,w) and (x,y) in units of (w,h)  (LAF.py:407-429).
 *   - fixed-capacity outputs: rows >= count are unspecified; counts live in device int32 arrays.
 */
#ifndef AFFNET_B200_H
#define AFFNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AG_OK 0
#define AG_ERR_INVALID -1   /* bad argument */
#define AG_ERR_CUDA -2      /* a CUDA runtime call failed */
#define AG_ERR_CAPACITY -3  /* a fixed-capacity buffer is too small */
#define AG_ERR_NO_DEVICE -4 /* no sm_100 device / kernel image not loadable */

#define AG_MAX_OCTAVES 16
#define AG_MAX_LEVELS 8 /* nlevels + 2 */

const char* ag_last_error(void);
/* ABI version of this header; bumps when a signature changes. */
int ag_abi_version(void);

/* Per-launch CUDA-event profiler (used by bench.py for the roofline leg; new, no reference counterpart).
 * Between ag_prof_begin(stream) and ag_prof_end() every kernel the library launches is followed by an event
 * record on `stream`; ag_prof_end() synchronises and returns the number of launches (or <0), ag_prof_get(i)
 * the name and duration in ms of launch i. */
int ag_prof_begin(void* stream);
int ag_prof_end(void);
int ag_prof_get(int i, const char** name, float* ms);

/* ------------------------------------------------------------------------------------------
 * Scale pyramid                   replaces ScalePyramid.forward  (HandCraftedModules.py:13-56)
 *                                 and GaussianBlur               (Utils.py:92-114,150-166)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int B, H, W;
    int n_octaves;
    int n_levels;                                        /* nlevels + 2 maps per octave */
    int h[AG_MAX_OCTAVES], w[AG_MAX_OCTAVES];            /* ceil-halved sizes (Q6) */
    long long level_offset[AG_MAX_OCTAVES][AG_MAX_LEVELS]; /* in floats from the pyramid base; each level is [B,h,w] */
    long long total_floats;
    double sigma[AG_MAX_OCTAVES][AG_MAX_LEVELS];         /* sigmas[o][l] of the reference (python floats) */
    double blur_sigma[AG_MAX_OCTAVES][AG_MAX_LEVELS];    /* sigma of the blur that produces level l (0: decimation) */
    double pix_dist[AG_MAX_OCTAVES];                     /* 2^o */
} ag_pyramid_plan_t;

/* Host-only: sizes, sigmas and buffer offsets (HandCraftedModules.py:15-22, 23-56 loop logic). */
int ag_pyramid_plan(int B, int H, int W, int nlevels, double init_sigma, int border, ag_pyramid_plan_t* plan);

/* d_img [B,H,W] -> d_pyr (plan->total_floats floats). */
int ag_pyramid_build(const ag_pyramid_plan_t* plan, const float* d_img, float* d_pyr, void* stream);

/* One Gaussian blur exactly as GaussianBlur(sigma)(x): k=int(6 sigma+1)|1 taps at linspace(-k/2,k/2,k),
 * replicate padding (Utils.py:150-166).  d_in/d_out [B,h,w]. */
int ag_gaussian_blur(const float* d_in, float* d_out, int B, int h, int w, double sigma, void* stream);

/* ------------------------------------------------------------------------------------------
 * Hessian response                replaces HessianResp.forward   (HandCraftedModules.py:58-78)
 * out = max(|gxx*gyy - gxy^2| * sigma^4 - th, 0)   (clamp: SparseImgRepresenter.py:77-84)
 * ------------------------------------------------------------------------------------------ */
int ag_hessian_response(const float* d_in, float* d_out, int B, int h, int w, double sigma, float th, void* stream);

/* ------------------------------------------------------------------------------------------
 * Detector: 3x3x3 NMS + border + octave map + soft-argmax + compaction
 *                                 replaces NMS3dAndComposeA.forward (HandCraftedModules.py:222-291)
 *                                 and the loop of multiScaleDetector (SparseImgRepresenter.py:53-111)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int B;
    int cand_cap;              /* capacity of the candidate list per image */
    int n_level_slots;         /* n_octaves * (n_levels-2) detection levels */
    /* device buffers, caller-allocated (sizes in elements) */
    float* d_cand_val;         /* [B, cand_cap]   response after octave-map masking (may be negative, Q4) */
    uint32_t* d_cand_seq;      /* [B, cand_cap]   (level_slot << 27) | flat pixel index; 0xFFFFFFFF = dropped */
    float* d_cand_scyx;        /* [B, cand_cap, 3] normalised (scale, y, x) */
    float* d_cand_aux;         /* [B, cand_cap, 2] raw NMS value of the same pixel at the octave's detection levels 1 and 2 */
    int* d_cand_count;         /* [B]             number appended (may exceed cand_cap -> overflow) */
    int* d_level_pos;          /* [B, n_level_slots] count of responses > 0 at each detection level */
    int* d_level_emit;         /* [B, n_level_slots] count of non-zero responses at each level */
    int* d_variants;           /* [B, n_octaves, 16] acceptance-hypothesis counters of the fused detector */
    uint8_t* d_octave_maps;    /* [4 * B * sum_o h_o*w_o] scratch for the octave maps (uint8, Q4 semantics) */
} ag_detect_ws_t;

/* Bytes needed for each workspace member are fixed by the struct comments; helper for callers: */
size_t ag_detect_ws_bytes(const ag_pyramid_plan_t* plan, int cand_cap);
/* Carves `d_ws` (ag_detect_ws_bytes bytes, 256-B aligned) into the struct's pointers. */
int ag_detect_ws_carve(const ag_pyramid_plan_t* plan, int cand_cap, void* d_ws, ag_detect_ws_t* ws);

/* All octaves/levels, Hessian fused (responses never touch HBM).  mr_border = int(mrSize). */
int ag_detect(const ag_pyramid_plan_t* plan, const float* d_pyr, float th, int mr_border, ag_detect_ws_t* ws, void* stream);

/* One detection level from precomputed response maps (B=1), for stage-isolated parity:
 * d_low/d_cur/d_high [h,w]; d_omap_in / d_omap_out uint8 [h,w] (in may be NULL = zeros).
 * Appends to ws (level slot `slot`), exactly like NMS3dAndComposeA given the same maps. */
int ag_detect_level_from_responses(const float* d_low, const float* d_cur, const float* d_high, int h, int w,
                                   const double scales[3], int mr_border, const uint8_t* d_omap_in,
                                   uint8_t* d_omap_out, int slot, ag_detect_ws_t* ws, void* stream);

/* Global selection (SparseImgRepresenter.py:100-111 + per-level rule HandCraftedModules.py:252-263):
 * levels with <=1 positive response are dropped; if more than num_features candidates remain the
 * top num_features by (response desc, seq asc) are returned sorted, otherwise all in
 * (octave, level, raster) order.  num_features <= 0 returns everything (capacity permitting).
 * a_scale multiplies the A part of the LAF (mrSize; SparseImgRepresenter.py:198).
 * Outputs [B, out_cap(,..)]: resp, LAFs (normalised), octave idx, level idx (= detection level-1); d_count[b] = -1 if the
 * candidate list of image b overflowed ws->cand_cap (the caller should retry with a larger capacity). */
int ag_select_keypoints(const ag_pyramid_plan_t* plan, const ag_detect_ws_t* ws, int num_features, float a_scale,
                        int out_cap, float* d_resp, float* d_lafs, int* d_oct, int* d_lvl, int* d_count,
                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Affine bilinear sampler          replaces extract_patches / generate_patch_grid_from_normalized_LAFs
 *                                  (LAF.py:313-372) and extract_patches_from_pyramid_with_inv_index
 *                                  (LAF.py:376-404)
 * out[n,c,i,j] = bilinear(img, p-0.5), p = A*min(h,w)*(xj,yi) + (x*w, y*h), xj=(2j+1)/PS-1, zeros outside
 * ------------------------------------------------------------------------------------------ */
/* Single image [C,h,w] (or per-patch images [n,C,h,w] when per_patch_img != 0), LAFs [n,2,3] normalised. */
int ag_extract_patches(const float* d_img, int C, int h, int w, int per_patch_img, const float* d_lafs, int n,
                       int PS, float* d_out, void* stream);

/* From the pyramid: image b of the batch, LAF i sampled at pyr[oct[i]][lvl[i]].  d_lafs [B,cap,2,3],
 * d_oct/d_lvl [B,cap], d_count [B] (NULL => all `cap` rows valid), d_out [B,cap,PS,PS]. */
int ag_extract_patches_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                           const int* d_lvl, const int* d_count, int cap, int PS, float* d_out, void* stream);

/* get_pyramid_and_level_index_for_LAFs (LAF.py:450-472): float64 argmin of |sigma_l*2^o - sqrt(|det A|+1e-12)/PS|.
 * d_dlafs [n,2,3] in pixel units. */
int ag_pyramid_level_for_lafs(const ag_pyramid_plan_t* plan, const float* d_dlafs, int n, int PS, int* d_oct,
                              int* d_lvl, void* stream);

/* ------------------------------------------------------------------------------------------
 * The three CNNs                    replaces AffNetFast.forward (architectures.py:204-252),
 *                                   OriNetFast.forward (architectures.py:33-82), HardNet.forward (HardNet.py:61-101)
 * ------------------------------------------------------------------------------------------ */
#define AG_NET_AFFNET 0
#define AG_NET_ORINET 1
#define AG_NET_HARDNET 2

typedef struct ag_net ag_net_t;

/* h_blob: the checkpoint tensors flattened in state_dict order without num_batches_tracked:
 * for each of the 6 conv layers: weight[Cout,Cin,3,3], running_mean[Cout], running_var[Cout];
 * then features.19.weight[Cout,Cin,8,8]; then bias[Cout] (AffNet, OriNet) or running_mean, running_var (HardNet).
 * BatchNorm (affine=False, eps 1e-5) is folded into the conv weights at upload. */
int ag_net_create(int kind, const float* h_blob, size_t n_floats, ag_net_t** out);
void ag_net_destroy(ag_net_t* net);
size_t ag_net_blob_floats(int kind);
/* Compute engine: 0 = exact fp32 SIMT (needs materialised patches);
 * 4 = tcgen05 tensor-core engine, THE DEFAULT for all three nets: fp16 operands, fp32 accumulation in TMEM, all six conv layers and the
 * 8x8 heads as MMAs; 128-pixel row tiles without x padding, the three taps of a kernel row stacked along N of one MMA, x shifts by warp
 * shuffles in the epilogue.  AffNet and OriNet carry fp16 residual planes of weights AND activations in every layer (fp32-grade: A 1e-5,
 * angle 3e-5 rad - OriNet's atan2 amplifies an error of AffNet's A about 15x, so the 1e-3 LAF contract needs A to 5e-5); HardNet fp16
 * activations with fp16 residuals of its layer 2-3 weights (descriptors 4e-4);
 * 5 = engine 4 with bf16 operands (HardNet only; BASELINE.json configs[4] "bf16 HardNet tensor-core path"; descriptors ~4e-3).
 * Engines 1, 2 and 3 (the first-generation tensor-core engine and its variants) no longer exist and are refused with AG_ERR_INVALID. */
int ag_net_set_engine(ag_net_t* net, int engine);
int ag_net_get_engine(const ag_net_t* net);
/* Developer switch: 1 = conv layer 3 of AffNet / OriNet runs inside the first tcgen05 kernel (layer 2's output stays in shared memory;
 * bit-identical; the default unless built with -DAG_FUSE_L3=0), 0 = first kernel and layer-3 kernel as two launches.  Returns the
 * previous mode. */
int ag_debug_fuse_l3(int fused);
/* Developer diagnostic: run the tensor-core trunk on materialised patches [n,32,32] up to conv layer `upto` (2..5) and decode
 * that layer's activations (fp16 hi [+ lo] planes in the engine's HBM layout) to fp32 [n,C,H,H].  d_ws: ag_net_workspace_bytes(). */
int ag_debug_tcx_layer(const ag_net_t* net, const float* d_patches, int n, int upto, float* d_out, void* d_ws, size_t ws_bytes, void* stream);
/* Scratch bytes for a forward over n patches. */
size_t ag_net_workspace_bytes(int kind, int n);

/* d_patches [n,1,32,32] (any scale: per-patch mean/std normalisation is part of forward).
 * Row validity: rows are grouped in groups of `group` rows (group <= 0 => one group of n rows); if d_count is
 * not NULL, only the first d_count[g] rows of group g are computed (device int32 array), else all rows.
 * AffNet -> d_out [n,2,2] rectified A.   OriNet -> d_out [n,2,2] rotation (and/or d_angle [n]; either may be NULL).
 * HardNet -> d_out [n,128] L2-normalised. */
int ag_affnet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out,
                      void* d_ws, size_t ws_bytes, void* stream);
int ag_orinet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out,
                      float* d_angle, void* d_ws, size_t ws_bytes, void* stream);
int ag_hardnet_forward(const ag_net_t* net, const float* d_patches, int n, const int* d_count, int group, float* d_out,
                       void* d_ws, size_t ws_bytes, void* stream);

/* f4: the TorchScript exports' contract (convertJIT/AffNetJIT.pt, OriNetJIT.pt; convert_OriNet_and_AffNet_to_JIT.ipynb): the RAW head
 * outputs.  AffNet: xy + [1, 0, 1] = (1 + x0, x1, 1 + x2) -> d_raw [n,3] (architectures.py:228-230 before rectification);
 * OriNet: the mean over the 3x3 map of tanh(conv8x8) -> d_raw [n,2] = (sin-like, cos-like) (architectures.py:57-59,76).
 * Tensor-core engine (4) only. */
int ag_affnet_forward_raw(const ag_net_t* net, const float* d_patches, int n, float* d_raw, void* d_ws, size_t ws_bytes, void* stream);
int ag_orinet_forward_raw(const ag_net_t* net, const float* d_patches, int n, float* d_raw, void* d_ws, size_t ws_bytes, void* stream);
/* Fused sampler + net (tensor-core engine): LAF i of image b is sampled at pyr[oct][lvl] INSIDE the first tensor-core
 * layer (32x32 patches never touch HBM), then the net runs as above.  Layout as ag_extract_patches_pyr: d_lafs
 * [B,cap,2,3] normalised, d_oct/d_lvl [B,cap], d_count [B] or NULL.  d_out: [B*cap,2,2] (AffNet, OriNet) or [B*cap,128]. */
int ag_net_forward_pyr(const ag_net_t* net, const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                       const int* d_lvl, const int* d_count, int cap, float* d_out, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Keypoint geometry                 replaces getAffineShape's filter (SparseImgRepresenter.py:136-162,
 *                                   Utils.py:168-175, LAF.py:98-104), getOrientation's compose (:175),
 *                                   denormalizeLAFs / normalizeLAFs (LAF.py:407-429)
 * ------------------------------------------------------------------------------------------ */
/* Per image b (B images, `cap` rows each, d_count_in[b] valid):  new_LAF = [A*LAF_A, t]; keep where
 * 1/6 < |l1/(l2+1e-8)| < 6 and the LAF does not touch the boundary; if survivors > num_features keep the
 * top num_features by response (desc; ties by index) else all survivors in order.
 * Outputs are compacted: d_resp_out/d_lafs_out/d_oct_out/d_lvl_out [B,out_cap..], d_count_out [B]. */
int ag_affine_shape_filter(const float* d_A, const float* d_resp, const float* d_lafs, const int* d_oct,
                           const int* d_lvl, const int* d_count_in, int B, int cap, int num_features, int out_cap,
                           float* d_resp_out, float* d_lafs_out, int* d_oct_out, int* d_lvl_out, int* d_count_out,
                           void* stream);

/* LAF_A <- LAF_A * R  then (optionally) denormalise to pixels of a WxH image.  d_lafs [n,2,3] in/out. */
int ag_lafs_apply_rotation(float* d_lafs, const float* d_R, int n, void* stream);
int ag_lafs_scale(const float* d_in, float* d_out, int n, float a_coef, float x_coef, float y_coef, void* stream);
/* The 2x2 chain of the Baumberg iterations (SparseImgRepresenter.py:127-141, torch.bmm there): d_out [n,2,2] = d_A * d_B;
 * d_out [n,2,3] = [d_A * d_lafs[:, :, :2] | d_lafs[:, :, 2]]. */
int ag_mat2_compose(const float* d_A, const float* d_B, float* d_out, int n, void* stream);
int ag_lafs_left_multiply(const float* d_A, const float* d_lafs, float* d_out, int n, void* stream);
/* Output format of the reference's writers (hesaffBaum.py:46-48): replaces LAFs2ellT (LAF.py:35-51, bsvd2x2 :106-144).
 * d_lafs [n,2,3] in pixels -> d_ell [n,5] = (x, y, a, b, c) with a u^2 + 2 b u v + c v^2 = 1.  A LAF with a negative
 * determinant gives NaN, as in the reference. */
int ag_lafs_to_ell(const float* d_lafs, int n, float* d_ell, void* stream);

/* ------------------------------------------------------------------------------------------
 * Hand-crafted estimators (SURVEY.md §8f "next" rows): what the reference uses when OriNet / AffNet are None.
 *   ag_orientation_hist  replaces OrientationDetector.forward   (HandCraftedModules.py:133-192): 36-bin gradient histogram,
 *                        (0.33,0.34,0.33) smoothing, arg-max -> angle [n]
 *   ag_baumberg_shape    replaces AffineShapeEstimator.forward  (HandCraftedModules.py:81-132): second-moment matrix ->
 *                        inverse square root -> up-is-up rectified A [n,2,2]
 * d_patches [n,PS,PS] (3 <= PS <= 41); d_gk [PS,PS] = the module's Gaussian window: ag_circular_gauss_kernel(PS, sigma, h_out)
 * reproduces CircularGaussKernel (Utils.py:92-114; sigma <= 0 selects the default sigma^2 = 0.9 (PS/2)^2 / 2); the orientation
 * window is 10x that kernel, the Baumberg window uses sigma = (PS/2)/3.
 * ------------------------------------------------------------------------------------------ */
int ag_circular_gauss_kernel(int kernlen, double sigma, float* h_out);
int ag_orientation_hist(const float* d_patches, int n, int PS, const float* d_gk, float* d_angle, void* stream);
int ag_baumberg_shape(const float* d_patches, int n, int PS, const float* d_gk, float* d_A, void* stream);
/* The same estimators sampling their patches from the pyramid inside the kernel (PS x PS patches never reach HBM).  Layout as
 * ag_extract_patches_pyr: d_lafs [B,cap,2,3] normalised, d_oct/d_lvl [B,cap], d_count [B] (NULL => all rows); rows i >= d_count[b] are
 * neither read nor written.  The Gaussian window is derived from PS as the modules derive it.  3 <= PS <= 41.
 *   ag_orientation_hist_pyr = ag_extract_patches_pyr -> ag_orientation_hist -> (cos, sin) -> ag_lafs_apply_rotation, bit for bit:
 *                             d_angle [B,cap] and/or d_lafs_out [B,cap,2,3] = [LAF_A * R | t], R = [[c, s], [-s, c]]; either may be
 *                             NULL (not both); d_lafs_out may equal d_lafs (rotates in place).
 *   ag_baumberg_shape_pyr   = the n_iters loop of getAffineShape (SparseImgRepresenter.py:155-166) over ag_extract_patches_pyr ->
 *                             ag_baumberg_shape -> ag_mat2_compose -> ag_lafs_left_multiply, bit for bit, in one launch:
 *                             d_A [B,cap,2,2] = base_A (1 <= n_iters <= 64). */
int ag_orientation_hist_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                            const int* d_lvl, const int* d_count, int cap, int PS, float* d_angle, float* d_lafs_out, void* stream);
int ag_baumberg_shape_pyr(const ag_pyramid_plan_t* plan, const float* d_pyr, const float* d_lafs, const int* d_oct,
                          const int* d_lvl, const int* d_count, int cap, int PS, int n_iters, float* d_A, void* stream);

/* Descriptor matching (SURVEY.md §8f row 3).
 *   ag_distance_matrix replaces distance_matrix_vector (Losses.py:5-13): out[n1,n2] = sqrt(|a|^2 + |b|^2 - 2 a.b + 1e-6)
 *   ag_match_snn       replaces the SNN-ratio block of train_AffNet_test_on_graffity.py:292-298: nearest neighbour, then
 *                      `dist[:, idxs_in_2] = 100000` (all columns that are anybody's nearest neighbour), second minimum,
 *                      keep[i] = min/(second + 1e-8) <= ratio.   Outputs [n1]: d_idx2, d_min, d_second, d_keep (uint8). */
int ag_distance_matrix(const float* d_a, int n1, const float* d_b, int n2, int dim, float* d_out, void* stream);
size_t ag_match_snn_workspace_bytes(int n1, int n2);
int ag_match_snn(const float* d_desc1, int n1, const float* d_desc2, int n2, int dim, float ratio, void* d_ws, size_t ws_bytes, int* d_idx2,
                 float* d_min, float* d_second, unsigned char* d_keep, void* stream);

/* ------------------------------------------------------------------------------------------
 * Batched end-to-end pipeline (new; the reference processes one image at a time):
 * pyramid -> detect -> select(1.5K) -> sample -> AffNet -> filter(K) -> [sample -> OriNet -> rotate]
 * -> denormalise -> level select -> sample -> HardNet.       = ScaleSpaceAffinePatchExtractor.forward
 * (the default estimators; ag_pipeline_create_ex selects the others: AffNet or Baumberg x num_Baum_iters or no shape
 * stage, OriNet, histogram or no orientation)
 * + extract_patches_from_pyr + HardNet.forward (train_AffNet_test_on_graffity.py:255-260) for B images.
 * ------------------------------------------------------------------------------------------ */
typedef struct ag_pipeline ag_pipeline_t;

typedef struct {
    int B, H, W;
    int num_features;   /* K */
    int nlevels;        /* 3 */
    int border;         /* 5 */
    double init_sigma;  /* 1.6 */
    double mrSize;      /* 5.192 */
    int do_ori;         /* 1: OriNet orientation */
    int cand_cap;       /* candidate capacity per image (0 => H*W/8); on overflow the image's count is reported as -1 */
} ag_pipeline_config_t;

/* Nets are borrowed (must outlive the pipeline).  The pipeline owns no device memory: the caller passes one
 * workspace of ag_pipeline_workspace_bytes() bytes.  Same as ag_pipeline_create_ex(cfg, NULL, ...). */
int ag_pipeline_create(const ag_pipeline_config_t* cfg, const ag_net_t* affnet, const ag_net_t* orinet,
                       const ag_net_t* hardnet, ag_pipeline_t** out);

/* Estimator configuration of the pipeline: the choices of ScaleSpaceAffinePatchExtractor's constructor
 * (SparseImgRepresenter.py:14-49) for the affine shape and orientation stages.
 *   shape          AG_SHAPE_AFFNET: num_Baum_iters AffNet iterations (sampler fused into the net), needs `affnet`;
 *                  AG_SHAPE_BAUMBERG: num_Baum_iters Baumberg iterations (AffineShapeEstimator) in one ag_baumberg_shape_pyr launch.
 *   num_Baum_iters 0..64; 0 = no shape stage: the K strongest keypoints go straight from the detector to orientation.
 *                  With 1 or more iterations int(1.5 K) keypoints are selected and the shape filter keeps K.
 *   shape_ps       patch size of the Baumberg estimator (3..41; 19 in the reference); ignored for AffNet (32).
 *   ori            AG_ORI_NONE; AG_ORI_ORINET (needs `orinet`); AG_ORI_HIST: gradient-histogram OrientationDetector,
 *                  one ag_orientation_hist_pyr launch.
 *   ori_ps         patch size of the histogram orientation (3..41; 19 in the reference); ignored otherwise.
 * est == NULL gives AG_SHAPE_AFFNET with 1 iteration and cfg->do_ori ? AG_ORI_ORINET : AG_ORI_NONE (ag_pipeline_create).
 * With est != NULL, est->ori governs and cfg->do_ori is ignored.  Invalid combinations fail here with AG_ERR_INVALID. */
#define AG_SHAPE_AFFNET 0
#define AG_SHAPE_BAUMBERG 1
#define AG_ORI_NONE 0
#define AG_ORI_ORINET 1
#define AG_ORI_HIST 2
typedef struct {
    int shape;           /* AG_SHAPE_* */
    int num_Baum_iters;  /* 0..64 */
    int shape_ps;        /* Baumberg patch size */
    int ori;             /* AG_ORI_* */
    int ori_ps;          /* histogram-orientation patch size */
} ag_pipeline_estimators_t;
int ag_pipeline_create_ex(const ag_pipeline_config_t* cfg, const ag_pipeline_estimators_t* est, const ag_net_t* affnet,
                          const ag_net_t* orinet, const ag_net_t* hardnet, ag_pipeline_t** out);
void ag_pipeline_destroy(ag_pipeline_t* p);
size_t ag_pipeline_workspace_bytes(const ag_pipeline_t* p);
const ag_pyramid_plan_t* ag_pipeline_plan(const ag_pipeline_t* p);
/* d_img [B,H,W] -> d_lafs [B,K,2,3] (pixel units), d_resp [B,K], d_desc [B,K,128], d_count [B].
 * Enqueues kernels only (CUDA-graph capturable). */
int ag_pipeline_run(ag_pipeline_t* p, const float* d_img, void* d_ws, size_t ws_bytes, float* d_lafs, float* d_resp,
                    float* d_desc, int* d_count, void* stream);
/* Number of kernel launches one ag_pipeline_run enqueues (for bench.py's gpu_launches). */
int ag_pipeline_launch_count(const ag_pipeline_t* p);

#ifdef __cplusplus
}
#endif
#endif /* AFFNET_B200_H */
