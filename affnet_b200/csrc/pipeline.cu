// Batched end-to-end pipeline: ScaleSpaceAffinePatchExtractor.forward (SparseImgRepresenter.py:189-209) + extract_patches_from_pyr
// (:181-188) + HardNet.forward for B images of one size, as a fixed sequence of kernel launches on one stream with fixed-capacity
// buffers and device-side counters (no host synchronisation, CUDA-graph capturable).  The reference processes one image at a time with
// several .item()/nonzero host round trips (SURVEY.md §3); this is the B200-native replacement.  The estimator stages follow the
// reference's constructor choices (ag_pipeline_estimators_t): AffNet or Baumberg x num_Baum_iters or none, OriNet or histogram or none.
#include "common.cuh"

struct ag_pipeline {
    ag_pipeline_config_t cfg;
    ag_pyramid_plan_t plan;
    const ag_net_t* aff;
    const ag_net_t* ori;
    const ag_net_t* hard;
    ag_pipeline_estimators_t est;
    int M;          // prefilter keypoints per image: int(1.5 K) with a shape stage, else K
    int cand_cap;
    // workspace layout (byte offsets); off_lafsw / off_A2 / off_Anet (working LAFs, second base_A, AffNet output) only for AffNet x n > 1
    size_t off_pyr, off_det, off_resp1, off_lafs1, off_oct1, off_lvl1, off_cnt1, off_patches, off_A, off_lafs2, off_oct2,
        off_lvl2, off_nlafs, off_oct3, off_lvl3, off_net, net_bytes, off_lafsw, off_A2, off_Anet, total;
    int launches;
};

using namespace ag;

extern "C" {

int ag_pipeline_create_ex(const ag_pipeline_config_t* cfg, const ag_pipeline_estimators_t* est, const ag_net_t* affnet,
                          const ag_net_t* orinet, const ag_net_t* hardnet, ag_pipeline_t** out) {
    AG_REQUIRE(cfg && hardnet && out, "NULL argument");
    AG_REQUIRE(cfg->num_features >= 1, "num_features must be positive");
    ag_pipeline_estimators_t e;
    if (est) {
        e = *est;
    } else {
        e.shape = AG_SHAPE_AFFNET; e.num_Baum_iters = 1; e.shape_ps = 32;
        e.ori = cfg->do_ori ? AG_ORI_ORINET : AG_ORI_NONE; e.ori_ps = 32;
    }
    AG_REQUIRE(e.shape == AG_SHAPE_AFFNET || e.shape == AG_SHAPE_BAUMBERG, "unknown shape estimator (AG_SHAPE_AFFNET or AG_SHAPE_BAUMBERG)");
    AG_REQUIRE(e.ori == AG_ORI_NONE || e.ori == AG_ORI_ORINET || e.ori == AG_ORI_HIST, "unknown orientation estimator (AG_ORI_NONE, AG_ORI_ORINET or AG_ORI_HIST)");
    AG_REQUIRE(e.num_Baum_iters >= 0 && e.num_Baum_iters <= 64, "num_Baum_iters out of range (0..64)");
    AG_REQUIRE(!(e.shape == AG_SHAPE_AFFNET && e.num_Baum_iters > 0) || affnet, "AG_SHAPE_AFFNET with num_Baum_iters > 0 needs an AffNet");
    AG_REQUIRE(!(e.shape == AG_SHAPE_BAUMBERG && e.num_Baum_iters > 0) || (e.shape_ps >= 3 && e.shape_ps <= 41),
               "Baumberg patch size out of range (3..41)");
    AG_REQUIRE(e.ori != AG_ORI_ORINET || orinet, "AG_ORI_ORINET needs an OriNet");
    AG_REQUIRE(e.ori != AG_ORI_HIST || (e.ori_ps >= 3 && e.ori_ps <= 41), "orientation patch size out of range (3..41)");
    ag_pipeline* p = new ag_pipeline();
    p->cfg = *cfg; p->est = e; p->aff = affnet; p->ori = orinet; p->hard = hardnet;
    int rc = ag_pyramid_plan(cfg->B, cfg->H, cfg->W, cfg->nlevels, cfg->init_sigma, cfg->border, &p->plan);
    if (rc != AG_OK) { delete p; return rc; }
    p->M = e.num_Baum_iters > 0 ? (int)(1.5 * cfg->num_features) : cfg->num_features;  // SparseImgRepresenter.py:44, 194
    if (p->M > 16384) {   // the selection kernels sort in shared memory (ag_select_keypoints / ag_affine_shape_filter): fail here, not at run time
        if (e.num_Baum_iters > 0)
            set_error("ag_pipeline_create: num_features %d needs a prefilter of int(1.5 K) = %d keypoints; the shared-memory selection holds 16384 (K <= 10922)",
                      cfg->num_features, p->M);
        else
            set_error("ag_pipeline_create: num_features %d: the shared-memory selection holds 16384 keypoints", cfg->num_features);
        delete p;
        return AG_ERR_CAPACITY;
    }
    p->cand_cap = cfg->cand_cap > 0 ? cfg->cand_cap : (cfg->H * cfg->W) / 8;
    if (p->cand_cap < p->M) p->cand_cap = p->M;
    const size_t B = cfg->B, M = p->M, K = cfg->num_features;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 256); return r; };
    p->off_pyr = take(sizeof(float) * (size_t)p->plan.total_floats);
    p->off_det = take(ag_detect_ws_bytes(&p->plan, p->cand_cap));
    p->off_resp1 = take(sizeof(float) * B * M);
    p->off_lafs1 = take(sizeof(float) * B * M * 6);
    p->off_oct1 = take(sizeof(int) * B * M);
    p->off_lvl1 = take(sizeof(int) * B * M);
    p->off_cnt1 = take(sizeof(int) * B);
    p->off_patches = 0;  // 32x32 patches are never materialised: the sampler is fused into the first tensor-core layer
    p->off_A = take(sizeof(float) * B * M * 4);
    p->off_lafs2 = take(sizeof(float) * B * K * 6);
    p->off_oct2 = take(sizeof(int) * B * K);
    p->off_lvl2 = take(sizeof(int) * B * K);
    p->off_nlafs = take(sizeof(float) * B * K * 6);
    p->off_oct3 = take(sizeof(int) * B * K);
    p->off_lvl3 = take(sizeof(int) * B * K);
    size_t nb = ag_net_workspace_bytes(AG_NET_AFFNET, (int)(B * M));
    size_t hb = ag_net_workspace_bytes(AG_NET_HARDNET, (int)(B * K));
    p->net_bytes = nb > hb ? nb : hb;
    p->off_net = take(p->net_bytes);
    p->off_lafsw = p->off_A2 = p->off_Anet = 0;
    if (e.shape == AG_SHAPE_AFFNET && e.num_Baum_iters > 1) {
        p->off_lafsw = take(sizeof(float) * B * M * 6);
        p->off_A2 = take(sizeof(float) * B * M * 4);
        p->off_Anet = take(sizeof(float) * B * M * 4);
    }
    p->total = o;
    p->launches = 0;
    *out = p;
    return AG_OK;
}

int ag_pipeline_create(const ag_pipeline_config_t* cfg, const ag_net_t* affnet, const ag_net_t* orinet, const ag_net_t* hardnet,
                       ag_pipeline_t** out) {
    return ag_pipeline_create_ex(cfg, nullptr, affnet, orinet, hardnet, out);
}

void ag_pipeline_destroy(ag_pipeline_t* p) { delete p; }
size_t ag_pipeline_workspace_bytes(const ag_pipeline_t* p) { return p ? p->total : 0; }
const ag_pyramid_plan_t* ag_pipeline_plan(const ag_pipeline_t* p) { return p ? &p->plan : nullptr; }
int ag_pipeline_launch_count(const ag_pipeline_t* p) { return p ? p->launches : 0; }

int ag_pipeline_run(ag_pipeline_t* p, const float* d_img, void* d_ws, size_t ws_bytes, float* d_lafs, float* d_resp,
                    float* d_desc, int* d_count, void* stream) {
    AG_REQUIRE(p && d_img && d_ws && d_lafs && d_resp && d_desc && d_count, "NULL argument");
    if (ws_bytes < p->total) {
        set_error("ag_pipeline_run: workspace of %zu bytes needed, %zu given", p->total, ws_bytes);
        return AG_ERR_CAPACITY;
    }
    char* ws = (char*)d_ws;
    const ag_pipeline_config_t& c = p->cfg;
    const int B = c.B, M = p->M, K = c.num_features;
    float* pyr = (float*)(ws + p->off_pyr);
    float* resp1 = (float*)(ws + p->off_resp1); float* lafs1 = (float*)(ws + p->off_lafs1);
    int* oct1 = (int*)(ws + p->off_oct1); int* lvl1 = (int*)(ws + p->off_lvl1); int* cnt1 = (int*)(ws + p->off_cnt1);
    float* A = (float*)(ws + p->off_A);
    float* lafs2 = (float*)(ws + p->off_lafs2); int* oct2 = (int*)(ws + p->off_oct2); int* lvl2 = (int*)(ws + p->off_lvl2);
    float* nlafs = (float*)(ws + p->off_nlafs); int* oct3 = (int*)(ws + p->off_oct3); int* lvl3 = (int*)(ws + p->off_lvl3);
    void* netws = ws + p->off_net;
    const int launches0 = g_launches;
    int rc;
    ag_detect_ws_t det;
    if ((rc = ag_detect_ws_carve(&p->plan, p->cand_cap, ws + p->off_det, &det))) return rc;
    if ((rc = ag_pyramid_build(&p->plan, d_img, pyr, stream))) return rc;
    if ((rc = ag_detect(&p->plan, pyr, 0.f, (int)c.mrSize, &det, stream))) return rc;
    const ag_pipeline_estimators_t& e = p->est;
    if (e.num_Baum_iters == 0) {
        // no shape stage (SparseImgRepresenter.py:207-211): the K strongest keypoints go straight to orientation
        if ((rc = ag_select_keypoints(&p->plan, &det, K, (float)c.mrSize, K, d_resp, lafs2, oct2, lvl2, d_count, stream))) return rc;
    } else {
        if ((rc = ag_select_keypoints(&p->plan, &det, M, (float)c.mrSize, M, resp1, lafs1, oct1, lvl1, cnt1, stream))) return rc;
        // affine shape: num_Baum_iters iterations of getAffineShape (SparseImgRepresenter.py:155-166) -> base_A
        const float* baseA = A;
        if (e.shape == AG_SHAPE_BAUMBERG) {
            if ((rc = ag_baumberg_shape_pyr(&p->plan, pyr, lafs1, oct1, lvl1, cnt1, M, e.shape_ps, e.num_Baum_iters, A, stream))) return rc;
        } else {
            float* A2 = (float*)(ws + p->off_A2); float* Anet = (float*)(ws + p->off_Anet); float* lafsw = (float*)(ws + p->off_lafsw);
            const float* cur = lafs1;
            for (int it = 0; it < e.num_Baum_iters; it++) {
                float* Aout = it == 0 ? A : Anet;
                if ((rc = ag_net_forward_pyr(p->aff, &p->plan, pyr, cur, oct1, lvl1, cnt1, M, Aout, netws, p->net_bytes, stream))) return rc;
                if (it > 0) {   // base_A <- A base_A, into the other of the two base_A buffers
                    float* nb = baseA == A ? A2 : A;
                    if ((rc = ag_mat2_compose(Anet, baseA, nb, B * M, stream))) return rc;
                    baseA = nb;
                }
                if (it != e.num_Baum_iters - 1) {
                    if ((rc = ag_lafs_left_multiply(baseA, lafs1, lafsw, B * M, stream))) return rc;
                    cur = lafsw;
                }
            }
        }
        if ((rc = ag_affine_shape_filter(baseA, resp1, lafs1, oct1, lvl1, cnt1, B, M, K, K, d_resp, lafs2, oct2, lvl2, d_count, stream))) return rc;
    }
    if (e.ori == AG_ORI_ORINET) {
        if ((rc = ag_net_forward_pyr(p->ori, &p->plan, pyr, lafs2, oct2, lvl2, d_count, K, A, netws, p->net_bytes, stream))) return rc;
        if ((rc = ag_lafs_apply_rotation(lafs2, A, B * K, stream))) return rc;
    } else if (e.ori == AG_ORI_HIST) {
        if ((rc = ag_orientation_hist_pyr(&p->plan, pyr, lafs2, oct2, lvl2, d_count, K, e.ori_ps, nullptr, lafs2, stream))) return rc;
    }
    // denormalizeLAFs (LAF.py:407-417), then descriptor patches: level choice + normalizeLAFs (LAF.py:419-429)
    const float ms = (float)(c.H < c.W ? c.H : c.W);
    if ((rc = ag_lafs_scale(lafs2, d_lafs, B * K, ms, (float)c.W, (float)c.H, stream))) return rc;
    if ((rc = ag_pyramid_level_for_lafs(&p->plan, d_lafs, B * K, 32, oct3, lvl3, stream))) return rc;
    if ((rc = ag_lafs_scale(d_lafs, nlafs, B * K, 1.0f / ms, (float)(1.0 / (double)c.W), (float)(1.0 / (double)c.H), stream))) return rc;
    if ((rc = ag_net_forward_pyr(p->hard, &p->plan, pyr, nlafs, oct3, lvl3, d_count, K, d_desc, netws, p->net_bytes, stream))) return rc;
    p->launches = g_launches - launches0;
    return AG_OK;
}

}  // extern "C"
