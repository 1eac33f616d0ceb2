// Internal definition of the opaque ag_net_t handle shared by the fp32 SIMT engine (nets_simt.cu) and the
// tensor-core engine (nets_tcx.cu).
#pragma once
#include <cuda_fp16.h>

#include <vector>

#include "common.cuh"

#define AG_ENGINE_SIMT 0     /* exact fp32 direct convolution */
#define AG_ENGINE_TC2 4      /* tcgen05 engine (tcx_*.cuh): fp16 operands, fp32 accumulate in TMEM, kernel-row taps stacked along N, heads as tensor-core
                                GEMMs; AffNet / OriNet with fp16 residual planes of weights and activations (fp32-grade), HardNet with weight residuals
                                in layers 2-3 */
#define AG_ENGINE_TC2_BF16 5 /* HardNet only: engine 4 with bf16 operands (BASELINE.json configs[4]); descriptors ~4e-3 of the fp32 reference */

struct ag_net {
    int kind;
    int engine;
    float* d_w[6];     // fp32 [9][cin][cout], BN folded   (d_w[0] doubles as the [9][C] first-layer weights)
    float* d_b[6];     // fp32 [cout]  (BN shift)
    float* d_w1;       // == d_w[0]
    __half* d_wx[6];   // second-generation packs (tcx_pack_layer), layers 1..5
    __half* d_all_x;
    __half* d_wx_bf[6];   // HardNet: the same packs in bf16 (engine 5); storage type is 16 bits either way
    __half* d_headh_bf;
    __half* d_headh;   // head for the tensor-core GEMM, k = (pixel*C/8 + c/8)*8 + c%8: HardNet fp16 [8192/8][128][8]; AffNet / OriNet [4096/8][32 hi | 32 lo][8]
    float* d_head_w;   // AffNet [3][4096], OriNet w_eff[4096][18] (per-position shifted copies), HardNet [8192][128]
    float* d_head_b;   // AffNet bias[3], OriNet bias[2], HardNet {scale[128], shift[128]}
    float w_inv_scale[6];   // tensor-core layers: 1 / (power-of-two scale of d_wx[l]); [0] = layer 1 (scaled in the kernel)
    float head_inv_scale;   // AffNet / OriNet tensor-core head: 1 / (power-of-two scale of d_headh)
    float* d_all;      // fp32 allocation
    __half* d_all_h;   // fp16 allocation
};

#include "tcgen05.cuh"

namespace ag {
tc::FirstSrc tc_src_patches(const float* patches);
tc::FirstSrc tc_src_pyramid(const ag_pyramid_plan_t* p, const float* pyr, const float* lafs, const int* oct, const int* lvl, int cap);
int tc_headx_forward(const ag_net* net, const void* feat, int n, int group, const int* count, float* out, float* angle, cudaStream_t st, float* raw = nullptr);
size_t tc_headx_bytes(int n);
void tcx_pack_layer(const float* wf, int ci, int co, int stride, int nsplit, int sw, float scale, std::vector<__half>& out, int bf16 = 0);
int tcx_nsplit(int kind, int layer);
int tcx_split_w(int kind, int layer);
int tcx_stride(int layer);
size_t tcx_act_bytes(int n);
int tcx_trunk_affori(const ag_net* net, const tc::FirstSrc& src, int n, int group, const int* count, void* bufA, void* bufB, void* feat,
                     cudaStream_t st, int upto);
int tcx_trunk_hardnet(const ag_net* net, const tc::FirstSrc& src, int n, int group, const int* count, void* bufA, void* bufB, void* headbuf,
                      cudaStream_t st, int upto, int bf16 = 0);
int tc_hardnet_head(const ag_net* net, const void* headbuf, int n, int group, const int* count, float* out, cudaStream_t st, int bf16 = 0);
}  // namespace ag
