"""The batched pipeline's estimator modes (-m gpu): AffNet or Baumberg x num_Baum_iters or no shape stage, OriNet or gradient-histogram
or no orientation - the configurations of ScaleSpaceAffinePatchExtractor's constructor.  Contract: the batched pipeline gives the same
bits as the single-image mirror for the same modules and images, and the two pyramid-sampling hand-crafted kernels give the same bits as
the compositions of existing entry points they replace."""
import ctypes as C
import math

import pytest
import torch

import affnet_oracle as O
from helpers import gold, gray_from_rgb, load_weights

pytestmark = pytest.mark.gpu

DEV = "cuda"
W = load_weights()


@pytest.fixture(scope="module")
def L():
    import affnet_b200._lib as lib
    lib.lib()
    return lib


@pytest.fixture(scope="module")
def nets():
    from affnet_b200.architectures import AffNetFast, OriNetFast
    from affnet_b200.HardNet import HardNet
    a, o, h = AffNetFast(PS=32), OriNetFast(PS=32), HardNet()
    a.load_state_dict(W["affnet"]); o.load_state_dict(W["orinet"]); h.load_state_dict(W["hardnet"])
    return a.eval().to(DEV), o.eval().to(DEV), h.eval().to(DEV)


def crop_img():
    return gray_from_rgb(gold("graf_crop.npz")["rgb"])


def bits(t):
    """Bit pattern of a float32 tensor: equality here is bit identity, NaN included."""
    return t.contiguous().view(torch.int32)


def modules(nets, shape, ori):
    from affnet_b200.HandCraftedModules import AffineShapeEstimator, OrientationDetector
    aff, orin, _ = nets
    A = {"affnet": aff, "baumberg": AffineShapeEstimator(patch_size=19), None: None}[shape]
    R = {"orinet": orin, "hist": OrientationDetector(patch_size=19), "none": None}[ori]
    return A, R


# (shape estimator, num_Baum_iters, orientation)
CONFIGS = [("affnet", 1, "hist"), ("affnet", 2, "orinet"), ("affnet", 2, "none"), ("baumberg", 16, "hist"), ("baumberg", 16, "none"),
           ("baumberg", 1, "orinet"), (None, 0, "hist"), (None, 0, "none")]


@pytest.mark.parametrize("shape,n_iters,ori", CONFIGS, ids=["%s-%d-%s" % c for c in CONFIGS])
def test_pipeline_estimators_equal_single_image_api(L, nets, shape, n_iters, ori):
    from affnet_b200.pipeline import DetectDescribePipeline
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    hn = nets[2]
    A, R = modules(nets, shape, ori)
    do_ori = ori != "none"
    img = crop_img()
    imgs = torch.cat([img, img.flip(3), O.synthetic_image(img.size(2), img.size(3), 5)]).to(DEV)
    K = 300
    pipe = DetectDescribePipeline(3, img.size(2), img.size(3), A, hn, R, num_features=K, do_ori=do_ori, num_Baum_iters=n_iters)
    lafs, resp, desc, cnt = [t.clone() for t in pipe.run(imgs)]
    torch.cuda.synchronize()
    det = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=K, border=5, num_Baum_iters=n_iters, AffNet=A, OriNet=R)
    for b in range(3):
        dL, r = det(imgs[b:b + 1], do_ori=do_ori)
        d = hn(det.extract_patches_from_pyr(dL, PS=32))
        n = int(cnt[b])
        assert n == dL.size(0) and n > 0
        assert torch.equal(resp[b, :n], r) and torch.equal(lafs[b, :n], dL) and torch.equal(desc[b, :n], d), "image %d" % b
    pipe.capture()
    l2, r2, d2, c2 = pipe.replay(imgs)
    torch.cuda.synchronize()
    assert torch.equal(c2, cnt)
    for b in range(3):
        n = int(cnt[b])
        assert torch.equal(l2[b, :n], lafs[b, :n]) and torch.equal(r2[b, :n], resp[b, :n]) and torch.equal(d2[b, :n], desc[b, :n])


# ---- stage-isolated: the fused kernels against the compositions of existing entry points -------------------------------------------

def stage_inputs(L, cap=64, counts=(50, 37), seed=3):
    """B = 2 pyramid (graf crop + synthetic), [2, cap] random normalised LAFs of which some reach outside the image, random levels,
    counts shorter than cap; the rows past the counts hold NaN LAFs that no kernel may read."""
    from affnet_b200.HandCraftedModules import ScalePyramid
    img = crop_img()
    x = torch.cat([img, O.synthetic_image(img.size(2), img.size(3), 9)]).to(DEV)
    plan, buf = ScalePyramid(nLevels=3, init_sigma=1.6, border=5).build(x)
    g = torch.Generator().manual_seed(seed)
    n = 2 * cap
    th = torch.rand(n, generator=g) * 2 * math.pi
    s = 0.02 + 0.12 * torch.rand(n, generator=g)
    e = 0.6 + 0.8 * torch.rand(n, generator=g)
    lafs = torch.zeros(n, 2, 3)
    lafs[:, 0, 0] = s * e * torch.cos(th); lafs[:, 0, 1] = -s / e * torch.sin(th)
    lafs[:, 1, 0] = s * e * torch.sin(th); lafs[:, 1, 1] = s / e * torch.cos(th)
    lafs[:, :, 2] = -0.15 + 1.3 * torch.rand(n, 2, generator=g)          # ~40 % of the patches cross the image border
    lafs = lafs.view(2, cap, 2, 3)
    oct_ = torch.randint(0, plan.n_octaves, (2, cap), generator=g, dtype=torch.int32)
    lvl = torch.randint(0, plan.n_levels, (2, cap), generator=g, dtype=torch.int32)
    for b, c in enumerate(counts):
        lafs[b, c:] = float("nan")
    cnt = torch.tensor(counts, dtype=torch.int32)
    return plan, buf, lafs.to(DEV).contiguous(), oct_.to(DEV), lvl.to(DEV), cnt.to(DEV), cap, counts


def patches_pyr(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS):
    out = torch.zeros(plan.B, cap, PS, PS, device=DEV)
    L.check(L.lib().ag_extract_patches_pyr(C.byref(plan), L.ptr(buf), L.ptr(lafs), L.ptr(oct_), L.ptr(lvl), L.ptr(cnt), cap, PS,
                                           L.ptr(out), L.stream_ptr()))
    return out


def orientation_composed(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS):
    """ag_extract_patches_pyr -> ag_orientation_hist (OrientationDetector) -> torch.cos / torch.sin -> ag_lafs_apply_rotation."""
    from affnet_b200.HandCraftedModules import OrientationDetector
    from affnet_b200.SparseImgRepresenter import angles2A
    P = patches_pyr(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS).view(-1, 1, PS, PS)
    ang = OrientationDetector(patch_size=PS)(P)
    R = angles2A(ang).contiguous()
    rot = lafs.clone().view(-1, 2, 3)
    L.check(L.lib().ag_lafs_apply_rotation(L.ptr(rot), L.ptr(R), rot.size(0), L.stream_ptr()))
    return ang.view(plan.B, cap), rot.view(plan.B, cap, 2, 3)


def orientation_fused(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS, in_place=False):
    ang = torch.full((plan.B, cap), -7.0, device=DEV)
    out = lafs.clone()
    src = out if in_place else lafs
    L.check(L.lib().ag_orientation_hist_pyr(C.byref(plan), L.ptr(buf), L.ptr(src), L.ptr(oct_), L.ptr(lvl), L.ptr(cnt), cap, PS,
                                            None if in_place else L.ptr(ang), L.ptr(out), L.stream_ptr()))
    return ang, out


@pytest.mark.parametrize("PS", [19, 41])
def test_orientation_hist_pyr_equals_composition(L, PS):
    plan, buf, lafs, oct_, lvl, cnt, cap, counts = stage_inputs(L)
    ang_ref, rot_ref = orientation_composed(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS)
    ang, rot = orientation_fused(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS)
    _, rot_ip = orientation_fused(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS, in_place=True)
    torch.cuda.synchronize()
    for b, n in enumerate(counts):
        assert torch.equal(bits(ang[b, :n]), bits(ang_ref[b, :n]))
        assert torch.equal(bits(rot[b, :n]), bits(rot_ref[b, :n]))
        assert torch.equal(bits(rot_ip[b, :n]), bits(rot_ref[b, :n]))
        assert bool((ang[b, n:] == -7.0).all()) and torch.equal(bits(rot[b, n:]), bits(lafs[b, n:]))     # rows past the count untouched
    assert len(set(ang[0, :counts[0]].tolist())) > 5


def test_orientation_hist_pyr_all_36_bins(L):
    """One keypoint's LAF rotated in 1-degree steps over a linear ramp (a single dominant gradient direction): the arg-max bin takes all
    36 values, so the in-kernel cos / sin meet torch.cos / torch.sin at every angle the estimator can produce."""
    from affnet_b200.HandCraftedModules import ScalePyramid
    H = Wd = 160
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(Wd, dtype=torch.float32), indexing="ij")
    img = (0.7 * xx + 0.25 * yy).view(1, 1, H, Wd).to(DEV)
    plan, buf = ScalePyramid(nLevels=3, init_sigma=1.6, border=5).build(img)
    n = 360
    th = torch.arange(n, dtype=torch.float64) * math.pi / 180.0
    s = 0.12
    lafs = torch.zeros(1, n, 2, 3, dtype=torch.float64)
    lafs[0, :, 0, 0] = s * torch.cos(th); lafs[0, :, 0, 1] = -s * torch.sin(th)
    lafs[0, :, 1, 0] = s * torch.sin(th); lafs[0, :, 1, 1] = s * torch.cos(th)
    lafs[0, :, 0, 2] = 0.5; lafs[0, :, 1, 2] = 0.5
    lafs = lafs.float().to(DEV).contiguous()
    oct_ = torch.zeros(1, n, dtype=torch.int32, device=DEV)
    lvl = torch.ones(1, n, dtype=torch.int32, device=DEV)
    for PS in (19, 41):
        ang_ref, rot_ref = orientation_composed(L, plan, buf, lafs, oct_, lvl, None, n, PS)
        ang, rot = orientation_fused(L, plan, buf, lafs, oct_, lvl, None, n, PS)
        torch.cuda.synchronize()
        assert torch.unique(ang).numel() == 36, torch.unique(ang).numel()
        assert torch.equal(bits(ang), bits(ang_ref)) and torch.equal(bits(rot), bits(rot_ref))


def baumberg_composed(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS, n_iters):
    """The loop of getAffineShape (SparseImgRepresenter.py:155-166) over existing entry points: ag_extract_patches_pyr ->
    AffineShapeEstimator (ag_baumberg_shape) -> ag_mat2_compose -> ag_lafs_left_multiply."""
    from affnet_b200.HandCraftedModules import AffineShapeEstimator
    est = AffineShapeEstimator(patch_size=PS)
    lib = L.lib()
    n = plan.B * cap
    cur, base = lafs, None
    for i in range(n_iters):
        A = est(patches_pyr(L, plan, buf, cur, oct_, lvl, cnt, cap, PS).view(-1, 1, PS, PS))
        if base is None:
            base = A
        else:
            nb = torch.empty_like(A)
            L.check(lib.ag_mat2_compose(L.ptr(A), L.ptr(base), L.ptr(nb), n, L.stream_ptr()))
            base = nb
        if i != n_iters - 1:
            cur = torch.empty_like(lafs)
            L.check(lib.ag_lafs_left_multiply(L.ptr(base), L.ptr(lafs), L.ptr(cur), n, L.stream_ptr()))
    return base.view(plan.B, cap, 2, 2)


@pytest.mark.parametrize("PS", [19, 41])
@pytest.mark.parametrize("n_iters", [1, 16])
def test_baumberg_shape_pyr_equals_composition(L, PS, n_iters):
    plan, buf, lafs, oct_, lvl, cnt, cap, counts = stage_inputs(L)
    ref = baumberg_composed(L, plan, buf, lafs, oct_, lvl, cnt, cap, PS, n_iters)
    out = torch.full((plan.B, cap, 2, 2), -7.0, device=DEV)
    L.check(L.lib().ag_baumberg_shape_pyr(C.byref(plan), L.ptr(buf), L.ptr(lafs), L.ptr(oct_), L.ptr(lvl), L.ptr(cnt), cap, PS, n_iters,
                                          L.ptr(out), L.stream_ptr()))
    torch.cuda.synchronize()
    for b, n in enumerate(counts):
        assert torch.equal(bits(out[b, :n]), bits(ref[b, :n]))
        assert bool((out[b, n:] == -7.0).all())
        assert int(torch.isfinite(out[b, :n]).all(dim=(1, 2)).sum()) > n // 2


# ---- the reference's application check through the batched path -----------------------------------------------------------------

def test_graf_1_to_6_application_counts_batched(L, nets):
    """train_AffNet_test_on_graffity.py::test() (AffNet x 1, OriNet=None -> histogram orientation, K=3000) with graf img1 and img6 as one
    B = 2 batch: tentative / true counts within the bounds tests/test_gpu_parity.py::test_graf_1_to_6_application_counts[hcori] applies
    to the reference's golden 281 / 91."""
    from affnet_b200.HandCraftedModules import OrientationDetector
    from affnet_b200.Losses import match_snn
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, _, hn = nets
    z, f = gold("graf_match.npz"), gold("graf_full.npz")
    imgs = torch.cat([gray_from_rgb(f["rgb"]), gray_from_rgb(z["rgb6"])]).to(DEV)
    pipe = DetectDescribePipeline(2, imgs.size(2), imgs.size(3), aff, hn, OrientationDetector(patch_size=19), num_features=3000,
                                  do_ori=True, num_Baum_iters=1)
    lafs, resp, desc, cnt = pipe.run(imgs)
    pipe.check()
    n1, n2 = int(cnt[0]), int(cnt[1])
    assert n1 == int(z["hcori_n1"]) and n2 == int(z["hcori_n2"])
    L1, d1, L2, d2 = lafs[0, :n1], desc[0, :n1], lafs[1, :n2], desc[1, :n2]
    i1, i2, _, _ = match_snn(d1, d2, float(z["snn"]))
    _, keep, _ = O.gt_correspondences(L1[i1].cpu(), L2[i2].cpu(), torch.from_numpy(z["H1to6"]), float(z["px"]))
    tent, true = int(i1.numel()), int(keep.numel())
    print("\nbatched graf 1<->6 hcori: %d tentatives / %d true (reference %d / %d)" % (tent, true, int(z["hcori_tent"]), int(z["hcori_true"])))
    assert abs(tent - int(z["hcori_tent"])) <= max(4, 0.03 * int(z["hcori_tent"]))
    assert abs(true - int(z["hcori_true"])) <= max(6, 0.08 * int(z["hcori_true"]))


# ---- validation at construction --------------------------------------------------------------------------------------------------

def test_invalid_estimator_combinations_refused(L, nets):
    from affnet_b200.HandCraftedModules import AffineShapeEstimator, OrientationDetector
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, ori, hn = nets
    kw = dict(num_features=100)
    cases = [
        (dict(AffNet=aff, OriNet=ori, num_Baum_iters=65), "num_Baum_iters out of range"),
        (dict(AffNet=aff, OriNet=ori, num_Baum_iters=-1), "num_Baum_iters out of range"),
        (dict(AffNet=AffineShapeEstimator(patch_size=43), OriNet=ori, num_Baum_iters=16), "Baumberg patch size out of range"),
        (dict(AffNet=AffineShapeEstimator(patch_size=2), OriNet=ori, num_Baum_iters=1), "Baumberg patch size out of range"),
        (dict(AffNet=aff, OriNet=OrientationDetector(patch_size=42)), "orientation patch size out of range"),
        (dict(AffNet=aff, OriNet=OrientationDetector(patch_size=2)), "orientation patch size out of range"),
        (dict(AffNet=None, OriNet=ori, num_Baum_iters=1), "needs an AffNet"),
        (dict(AffNet=aff, OriNet=None, do_ori=True), "needs an OriNet"),
    ]
    for args, msg in cases:
        with pytest.raises(L.AffnetB200Error, match=msg):
            DetectDescribePipeline(1, 64, 80, HardNet=hn, **args, **kw)
    # valid edge cases construct
    DetectDescribePipeline(1, 64, 80, None, hn, OrientationDetector(patch_size=41), num_Baum_iters=0, **kw)
    DetectDescribePipeline(1, 64, 80, AffineShapeEstimator(patch_size=3), hn, None, do_ori=False, num_Baum_iters=64, **kw)
