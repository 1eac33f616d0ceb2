"""GPU parity tests (-m gpu): the CUDA path, called through the Python mirror -> C ABI, against the CPU oracle
on the same inputs.  Contract (SURVEY.md §8a Q7): (i) stage-isolated - NMS / selection / filters are identical
given identical inputs, float stages within stated tolerances; (ii) end to end - >=99.5 % keypoints matched,
matched LAFs / descriptors within 1e-3-level tolerances."""
import ctypes as C

import numpy as np
import pytest
import torch

import affnet_oracle as O
from helpers import TOL, gold, gray_from_rgb, laf_rel_errors, load_weights, match_keypoints, orientation_boundary_shares, parity_report

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


def pyr_to_flat(L, pyr, plan):
    buf = torch.zeros(plan.total_floats, dtype=torch.float32)
    for o in range(plan.n_octaves):
        for l in range(plan.n_levels):
            n = plan.h[o] * plan.w[o]
            buf[plan.level_offset[o][l]:plan.level_offset[o][l] + n] = pyr[o][l].reshape(-1)
    return buf.to(DEV)


def run_detect(L, plan, pyr_buf, nf, a_scale, mr=5, th=0.0, cap=None):
    lib = L.lib()
    cap = cap or max(plan.H * plan.W // 8, 4096)
    ws_buf = torch.empty(lib.ag_detect_ws_bytes(C.byref(plan), cap), dtype=torch.uint8, device=DEV)
    ws = L.DetectWs()
    L.check(lib.ag_detect_ws_carve(C.byref(plan), cap, L.ptr(ws_buf), C.byref(ws)))
    L.check(lib.ag_detect(C.byref(plan), L.ptr(pyr_buf), th, mr, C.byref(ws), L.stream_ptr()))
    resp = torch.empty(nf, device=DEV); lafs = torch.empty(nf, 2, 3, device=DEV)
    oc = torch.empty(nf, dtype=torch.int32, device=DEV); lv = torch.empty(nf, dtype=torch.int32, device=DEV)
    cnt = torch.empty(1, dtype=torch.int32, device=DEV)
    L.check(lib.ag_select_keypoints(C.byref(plan), C.byref(ws), nf, a_scale, nf, L.ptr(resp), L.ptr(lafs), L.ptr(oc), L.ptr(lv), L.ptr(cnt), L.stream_ptr()))
    n = int(cnt.item())
    return resp[:n].cpu(), lafs[:n].cpu(), oc[:n].cpu(), lv[:n].cpu(), ws, ws_buf


# ------------------------------------------------------------------------------------------------------------
def test_gaussian_blur_and_pyramid_vs_oracle(L):
    from affnet_b200.Utils import GaussianBlur
    from affnet_b200.HandCraftedModules import ScalePyramid
    g = torch.Generator().manual_seed(3)
    x = torch.rand(1, 1, 97, 131, generator=g) * 255
    for s in (1.5198684, 1.2262735, 1.5450078, 1.9465878, 2.4525304, 0.8, 3.3):
        d = (GaussianBlur(s)(x.to(DEV)).cpu() - O.gaussian_blur(x, s)).abs().max().item()
        assert d < 5e-4, (s, d)                     # 0..255 scale; separable fp32 vs dense fp32 (Q7: 2.6e-4)
    img = crop_img()
    pyr_o, sig_o, pix_o = O.scale_pyramid(img)
    pyr, sig, pix = ScalePyramid(3, 1.6, 5)(img.to(DEV))
    assert len(pyr) == len(pyr_o) and sig == sig_o and pix == pix_o
    worst = max((a.cpu() - b).abs().max().item() for oa, ob in zip(pyr, pyr_o) for a, b in zip(oa, ob))
    assert worst < 1e-3, worst
    # batch of 2 == two singles (bit exact)
    x2 = torch.cat([img, img.flip(3)]).to(DEV)
    p2, _, _ = ScalePyramid(3, 1.6, 5)(x2)
    assert torch.equal(p2[2][3][0], pyr[2][3][0])


def test_hessian_bit_exact(L):
    from affnet_b200.HandCraftedModules import HessianResp
    g = torch.Generator().manual_seed(4)
    for (h, w) in ((33, 70), (64, 64), (5, 7)):
        x = torch.rand(1, 1, h, w, generator=g) * 255
        x = O.gaussian_blur(x, 1.2)
        for s in (1.6, 2.0158736798317967, 3.1999999999999997):
            assert torch.equal(HessianResp()(x.to(DEV), s).cpu(), O.hessian_response(x, s))


def test_nms_level_identical_given_response_maps(L):
    """a4/a5 incl. the uint8-wrapping octave map (Q4): identical survivor set, values, map."""
    lib = L.lib()
    z = gold("nms_q4.npz")
    cases = [(z["low"], z["cur"], z["high"], z["omap"], list(z["scales"]))]
    g = torch.Generator().manual_seed(11)
    for (h, w) in ((37, 45), (64, 96), (12, 13)):
        maps = [O.gaussian_blur(torch.rand(1, 1, h, w, generator=g) * 500, 0.9)[0, 0].numpy() for _ in range(3)]
        om = (torch.rand(h, w, generator=g) * 3.2).byte().numpy()
        om[:, : w // 2] = 0
        cases.append((maps[0], maps[1], maps[2], om, [1.6, 2.0158736798317967, 2.5398416831491195]))
    for low, cur, high, om, scales in cases:
        h, w = cur.shape
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).view(1, 1, h, w)  # noqa: E731
        r_o, A_o, om_o, idx_o = O.nms3d_and_compose(t(low), t(cur), t(high), 0, om.copy(), scales, 5.192)
        plan = L.make_plan(1, h, w, 3, 1.6, 0)
        cap = h * w
        ws_buf = torch.zeros(lib.ag_detect_ws_bytes(C.byref(plan), cap), dtype=torch.uint8, device=DEV)
        ws = L.DetectWs()
        L.check(lib.ag_detect_ws_carve(C.byref(plan), cap, L.ptr(ws_buf), C.byref(ws)))
        d = [t(a).to(DEV).contiguous() for a in (low, cur, high)]
        om_in = torch.from_numpy(om).to(DEV).contiguous()
        om_out = torch.zeros_like(om_in)
        sc = (C.c_double * 3)(*scales)
        L.check(lib.ag_detect_level_from_responses(L.ptr(d[0]), L.ptr(d[1]), L.ptr(d[2]), h, w, sc, 5, L.ptr(om_in), L.ptr(om_out), 0,
                                                   C.byref(ws), L.stream_ptr()))
        nf = cap
        resp = torch.empty(nf, device=DEV); lafs = torch.empty(nf, 2, 3, device=DEV)
        oc = torch.empty(nf, dtype=torch.int32, device=DEV); lv = torch.empty(nf, dtype=torch.int32, device=DEV)
        cnt = torch.empty(1, dtype=torch.int32, device=DEV)
        if cap * 12 <= 200 * 1024:
            L.check(lib.ag_select_keypoints(C.byref(plan), C.byref(ws), 0, 1.0, nf, L.ptr(resp), L.ptr(lafs), L.ptr(oc), L.ptr(lv), L.ptr(cnt), L.stream_ptr()))
            n = int(cnt.item())
            if r_o is None:
                assert n == 0
            else:
                assert n == r_o.numel()
                assert torch.equal(resp[:n].cpu(), r_o)            # raster order, identical values (incl. negatives)
                assert (lafs[:n].cpu() - A_o).abs().max() < 1e-6
        if r_o is not None:
            assert np.array_equal(om_out.cpu().numpy(), om_o)
            # raw candidate list: same pixel set
            n_c = int(ws_buf[ws.d_cand_count - ws_buf.data_ptr():][:4].view(torch.int32).item())
            seq = ws_buf[ws.d_cand_seq - ws_buf.data_ptr():][:4 * n_c].view(torch.int32).cpu().numpy().astype(np.int64) & 0x7FFFFFF
            assert sorted(seq.tolist()) == sorted(idx_o.tolist())


def test_detector_identical_given_oracle_pyramid(L):
    """a3-a6 fused: feed the ORACLE's pyramid, demand the oracle's keypoints (set, order, values)."""
    img = crop_img()
    pyr, sig, pix = O.scale_pyramid(img)
    plan = L.make_plan(1, img.size(2), img.size(3), 3, 1.6, 5)
    buf = pyr_to_flat(L, pyr, plan)
    for nf in (450, 200, 4000):
        r_o, L_o, p_o, l_o = O.multi_scale_detector(pyr, sig, nf, 5.192)
        r, la, oc, lv, _, _ = run_detect(L, plan, buf, nf, 1.0)
        assert r.numel() == r_o.numel()
        assert torch.equal(r, r_o)
        assert torch.equal(oc.float(), p_o) and torch.equal(lv.float(), l_o)
        assert (la - L_o).abs().max() < 1e-6


def test_detector_threshold_mode_returns_all(L):
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    img = crop_img()[:, :, :128, :160].contiguous()
    det = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=100, border=5, num_Baum_iters=0, th=5.0)
    r, la, oc, lv = det.multiScaleDetector(img.to(DEV), det.num)
    pyr, sig, pix = O.scale_pyramid(img)
    # oracle with the same th, fed with OUR pyramid to isolate the stage
    pyr_g = [[t.cpu() for t in o] for o in det.scale_pyr]
    r_o, L_o, p_o, l_o = O.multi_scale_detector(pyr_g, sig, -1, 5.192, th=5.0)
    assert r.numel() == r_o.numel() and torch.equal(r.cpu(), r_o)
    assert torch.equal(oc.cpu(), p_o) and (la.cpu() - L_o).abs().max() < 1e-6


def test_sampler_vs_oracle(L):
    from affnet_b200.LAF import extract_patches
    g = torch.Generator().manual_seed(5)
    img = O.gaussian_blur(torch.rand(1, 1, 120, 150, generator=g) * 255, 1.0)
    n = 257
    lafs = torch.zeros(n, 2, 3)
    lafs[:, :, :2] = (torch.rand(n, 2, 2, generator=g) - 0.5) * 0.5
    lafs[:, :, 2] = torch.rand(n, 2, generator=g) * 1.4 - 0.2          # some patches leave the image
    for PS in (32, 19, 41):
        a = extract_patches(img.to(DEV), lafs.to(DEV), PS).cpu()
        b = O.extract_patches(img, lafs, PS)
        assert (a - b).abs().max() < 2e-2                               # 0..255 scale, fp32 coordinates x gradient
    rgb = torch.cat([img, img * 0.5, img.flip(2)], 1)
    a = extract_patches(rgb.to(DEV), lafs.to(DEV), 16).cpu()
    assert (a[:, 1] - 0.5 * a[:, 0]).abs().max() < 1e-4


def test_level_selection_identical(L):
    from affnet_b200.LAF import get_pyramid_and_level_index_for_LAFs
    z = gold("graf_crop.npz")
    plan = L.make_plan(1, z["rgb"].shape[0], z["rgb"].shape[1], 3, 1.6, 5)
    for tag in ("noori", "ori"):
        o, l = get_pyramid_and_level_index_for_LAFs(torch.from_numpy(z[tag + "_dLAFs"]).to(DEV), plan, 32)
        assert np.array_equal(o.cpu().numpy(), z[tag + "_desc_oct"]) and np.array_equal(l.cpu().numpy(), z[tag + "_desc_lvl"])
    g = torch.Generator().manual_seed(6)
    dl = torch.randn(5000, 2, 3, generator=g) * 40
    sizes, bs, sig, pix = O.pyramid_plan(*z["rgb"].shape[:2])
    oo, lo = O.pyramid_level_for_lafs(dl, sig, pix, 32)
    o, l = get_pyramid_and_level_index_for_LAFs(dl.to(DEV), plan, 32)
    assert torch.equal(o.cpu().float(), oo) and torch.equal(l.cpu().float(), lo)


@pytest.mark.parametrize("engine", ["simt"])
def test_nets_vs_oracle(L, nets, engine):
    """a9/a12/a16.  simt = exact fp32 engine (1e-4); the default tensor-core engine has its own checks in tests/test_gpu_tcx.py."""
    aff, ori, hn = nets
    z = gold("graf_crop.npz")
    g = torch.Generator().manual_seed(8)
    sets = [torch.from_numpy(z["aff_patches"]), torch.from_numpy(z["ori_desc_patches"]), torch.rand(37, 1, 32, 32, generator=g) * 255,
            torch.from_numpy(gold("face_patches.npz")["patches_u8"].astype(np.float32) / 255.0).view(-1, 1, 32, 32),
            torch.rand(300, 1, 32, 32, generator=g)]
    try:
        for m in (aff, ori, hn):
            m.set_engine(L.ENGINE_SIMT)
        worst = [0.0, 0.0, 0.0, 0.0]
        for P in sets:
            Pd = P.to(DEV)
            dA = (aff(Pd).cpu() - O.affnet_forward(P, W["affnet"])).abs().max().item()
            dR = (ori(Pd).cpu() - O.orinet_forward(P, W["orinet"])).abs().max().item()
            dang = (ori(Pd, return_rot_matrix=False).cpu() - O.orinet_angle(P, W["orinet"]))
            dang = torch.atan2(torch.sin(dang), torch.cos(dang)).abs().max().item()
            dD = (hn(Pd).cpu() - O.hardnet_forward(P, W["hardnet"])).abs().max().item()
            worst = [max(a, b) for a, b in zip(worst, (dA, dR, dang, dD))]
        print("\nengine %s: max|dA| %.2e  max|dR| %.2e  max|dangle| %.2e rad  max|ddesc| %.2e" % ((engine,) + tuple(worst)))
        assert max(worst) < 1e-4, worst
    finally:
        aff.set_engine(L.ENGINE_TC2); ori.set_engine(L.ENGINE_TC2); hn.set_engine(L.ENGINE_TC2)
    assert aff(torch.empty(0, 1, 32, 32, device=DEV)).shape == (0, 2, 2)


def test_nets_batching_invariance(L, nets):
    """Tile boundaries of the tensor-core path (2 patches per CTA pair, 128 per head tile, persistent strides over the SMs):
    every patch's result is bit-identical whatever batch it is evaluated in."""
    aff, ori, hn = nets
    g = torch.Generator().manual_seed(21)
    P = (torch.rand(513, 1, 32, 32, generator=g) * 255).to(DEV)
    for m in (aff, ori, hn):
        full = m(P)
        for lo, hi in ((0, 1), (1, 130), (130, 387), (386, 513), (512, 513)):
            assert torch.equal(m(P[lo:hi].contiguous()), full[lo:hi]), (type(m).__name__, lo, hi)


def test_shape_filter_identical_given_A(L):
    lib = L.lib()
    z = gold("graf_crop.npz")
    K = int(z["K"])
    Lf = torch.from_numpy(z["det_LAFs"]).clone(); Lf[:, 0:2, 0:2] = 5.192 * Lf[:, :, 0:2]
    A = torch.from_numpy(z["aff_A"]); resp = torch.from_numpy(z["det_resp"])
    n = A.size(0)
    for nf in (K, 50, 0):
        d = lambda t, dt=torch.float32: t.to(dt).to(DEV).contiguous()  # noqa: E731
        ro = torch.empty(n, device=DEV); lo = torch.empty(n, 2, 3, device=DEV)
        oo = torch.empty(n, dtype=torch.int32, device=DEV); vo = torch.empty(n, dtype=torch.int32, device=DEV)
        ci = torch.tensor([n], dtype=torch.int32, device=DEV); co = torch.empty(1, dtype=torch.int32, device=DEV)
        dA, dr, dL = d(A), d(resp), d(Lf)
        do, dv = d(torch.from_numpy(z["det_pidx"]), torch.int32), d(torch.from_numpy(z["det_lidx"]), torch.int32)
        L.check(lib.ag_affine_shape_filter(L.ptr(dA), L.ptr(dr), L.ptr(dL), L.ptr(do), L.ptr(dv), L.ptr(ci), 1, n, nf, n, L.ptr(ro), L.ptr(lo),
                                           L.ptr(oo), L.ptr(vo), L.ptr(co), L.stream_ptr()))
        m = int(co.item())
        newL = torch.cat([torch.bmm(A, Lf[:, :, :2]), Lf[:, :, 2:]], 2)
        mask = O.shape_filter_mask(A, newL)
        if nf > 0 and int(mask.sum()) > nf:
            r_o, idxs = torch.topk(resp * mask.float(), k=nf)
        else:
            idxs = mask.nonzero().view(-1); r_o = resp[idxs]
        assert m == r_o.numel() and torch.equal(ro[:m].cpu(), r_o)
        assert (lo[:m].cpu() - newL[idxs]).abs().max() < 1e-6
        if nf == K:
            assert torch.equal(ro[:m].cpu(), torch.from_numpy(z["shape_resp"]))     # the reference's own selection


@pytest.mark.parametrize("name,K", [("graf_crop.npz", 300), ("graf_full.npz", 2000)])
@pytest.mark.parametrize("do_ori", [False, True])
def test_end_to_end_vs_oracle(L, nets, name, K, do_ori):
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    aff, ori, hn = nets
    img = gray_from_rgb(gold(name)["rgb"])
    det = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=K, border=5, num_Baum_iters=1, AffNet=aff, OriNet=ori)
    with torch.no_grad():
        dL, resp = det(img.to(DEV), do_ori=do_ori)
        patches = det.extract_patches_from_pyr(dL, PS=32)
        desc = hn(patches)
    oL, oresp, st = O.detect(img, W["affnet"], W["orinet"], K, do_ori=do_ori)
    odesc, _, _ = O.describe(oL, st, W["hardnet"])
    assert dL.shape[0] == oL.shape[0] or abs(dL.shape[0] - oL.shape[0]) <= 0.005 * K
    ia, ib = match_keypoints(oL, dL.cpu())
    # >= 99.5 % (SURVEY Q7); the near-isotropic eigen-discriminant test of batch_eig2x2 flips ~1e-3 of the candidates under
    # any fp32 perturbation (the oracle itself differs from the reference by 2/3000 there), so allow 3 at small K
    assert len(ia) >= oL.shape[0] - max(3, 0.005 * oL.shape[0]), (len(ia), oL.shape[0])
    rep = parity_report(oL, odesc, dL.cpu(), desc.cpu(), "%s K=%d ori=%s vs oracle" % (name, K, do_ori))
    assert rep["eA"] < TOL and rep["ec"] < TOL and rep["dd"] < TOL, rep
    # the reference's own golden output, same contract
    z = gold(name)
    tag = "ori" if do_ori else "noori"
    gL = torch.from_numpy(z[tag + "_dLAFs"])
    rep = parity_report(gL, torch.from_numpy(z[tag + "_desc"]).float(), dL.cpu(), desc.cpu(), "%s K=%d ori=%s vs reference golden" % (name, K, do_ori))
    assert rep["matched"] >= gL.shape[0] - max(3, 0.005 * gL.shape[0])
    assert rep["eA"] < TOL and rep["ec"] < TOL and rep["dd"] < TOL, rep


def test_pipeline_batched_equals_single_image_api(L, nets):
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, ori, hn = nets
    img = crop_img()
    imgs = torch.cat([img, img.flip(3), O.synthetic_image(img.size(2), img.size(3), 5)]).to(DEV)
    K = 300
    for do_ori in (True, False):
        pipe = DetectDescribePipeline(3, img.size(2), img.size(3), aff, hn, ori, num_features=K, do_ori=do_ori)
        lafs, resp, desc, cnt = pipe.run(imgs)
        torch.cuda.synchronize()
        lafs, resp, desc, cnt = lafs.clone(), resp.clone(), desc.clone(), cnt.clone()
        assert pipe.launches > 30
        det = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=K, border=5, num_Baum_iters=1, AffNet=aff, OriNet=ori)
        for b in range(3):
            dL, r = det(imgs[b:b + 1], do_ori=do_ori)
            d = hn(det.extract_patches_from_pyr(dL, PS=32))
            n = int(cnt[b])
            assert n == dL.size(0)
            assert torch.equal(resp[b, :n], r) and torch.equal(lafs[b, :n], dL) and torch.equal(desc[b, :n], d)
        pipe.capture()
        l2, r2, d2, c2 = pipe.replay(imgs)
        torch.cuda.synchronize()
        assert torch.equal(c2, cnt)
        for b in range(3):
            n = int(cnt[b])
            assert torch.equal(l2[b, :n], lafs[b, :n]) and torch.equal(d2[b, :n], desc[b, :n])


def test_full_size_properties(L, nets):
    """BASELINE config 2 size (1024x768, K=2000): size-independent properties + oracle spot check."""
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, ori, hn = nets
    B, H, Wd, K = 2, 768, 1024, 2000
    imgs = torch.cat([O.synthetic_image(H, Wd, 1234 + i) for i in range(B)]).to(DEV)
    pipe = DetectDescribePipeline(B, H, Wd, aff, hn, ori, num_features=K, do_ori=True)
    lafs, resp, desc, cnt = [t.clone() for t in pipe.run(imgs)]
    l2, r2, d2, c2 = pipe.run(imgs)
    torch.cuda.synchronize()
    assert torch.equal(cnt, c2) and torch.equal(lafs, l2) and torch.equal(desc, d2)      # deterministic
    for b in range(B):
        n = int(cnt[b])
        assert 0 < n <= K
        r = resp[b, :n]
        assert bool((r[:-1] >= r[1:]).all()) and bool((r > 0).all())                     # sorted by response
        assert ((desc[b, :n].norm(dim=1) - 1).abs().max() < 1e-4)                         # L2-normalised
        c = lafs[b, :n, :, 2]
        assert bool((c[:, 0] >= 0).all() and (c[:, 0] <= Wd).all() and (c[:, 1] >= 0).all() and (c[:, 1] <= H).all())
    # candidate overflow is reported, not silently truncated
    small = DetectDescribePipeline(B, H, Wd, aff, hn, ori, num_features=K, do_ori=True, cand_cap=4000)
    small.run(imgs)
    with pytest.raises(Exception):
        small.check()
    oL, oresp, st = O.detect(imgs[0:1].cpu(), W["affnet"], W["orinet"], K, do_ori=True)
    odesc, _, _ = O.describe(oL, st, W["hardnet"])
    n = int(cnt[0])
    rep = parity_report(oL, odesc, lafs[0, :n].cpu(), desc[0, :n].cpu(), "synthetic 1024x768 K=2000 (bench workload) vs oracle")
    assert rep["matched"] >= 0.995 * oL.shape[0]
    assert rep["eA"] < TOL and rep["ec"] < TOL and rep["dd"] < TOL, rep


def _graf_1024():
    """SURVEY 8(d) input 2: graf img1 (800x640) resized to 1024x768 with cv2 INTER_LINEAR, then the channel mean of hesaffnet.py:35-39."""
    import cv2
    rgb = cv2.resize(gold("graf_full.npz")["rgb"], (1024, 768), interpolation=cv2.INTER_LINEAR)
    return gray_from_rgb(rgb)


@pytest.mark.parametrize("cfg", ["graf1024", "1080p", "4k"])
def test_benchmark_configs_vs_oracle(L, nets, cfg):
    """The configurations bench.py measures (BASELINE.json configs 2, 3, 5), one image each through the batched pipeline, against the
    oracle on the same image: >= 99.5 % of the keypoints matched, matched LAFs (relative to their scale) and descriptors within 1e-3."""
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, ori, hn = nets
    if cfg == "graf1024":
        img, K, border = _graf_1024(), 2000, 5
    elif cfg == "1080p":
        img, K, border = O.synthetic_image(1080, 1920, 1234), 4000, 5
    else:
        img, K, border = O.synthetic_image(2160, 3840, 4321), 8000, 33          # border=33 -> the 5-octave pyramid of config 5
    H, Wd = img.shape[2:]
    pipe = DetectDescribePipeline(1, H, Wd, aff, hn, ori, num_features=K, border=border, do_ori=True)
    lafs, resp, desc, cnt = pipe.run(img.to(DEV))
    pipe.check()
    n = int(cnt[0])
    torch.set_num_threads(min(16, torch.get_num_threads()))
    oL, oresp, st = O.detect(img, W["affnet"], W["orinet"], K, border=border, do_ori=True)
    odesc, _, _ = O.describe(oL, st, W["hardnet"])
    if cfg == "4k":
        assert len(st["pyr"]) == 5
    rep = parity_report(oL, odesc, lafs[0, :n].cpu(), desc[0, :n].cpu(), "%s K=%d border=%d vs oracle" % (cfg, K, border))
    assert abs(n - oL.shape[0]) <= 0.005 * K and rep["matched"] >= 0.995 * oL.shape[0], rep
    assert rep["eA"] < TOL and rep["ec"] < TOL and rep["dd"] < TOL, rep
    if cfg == "4k":      # BASELINE.json configs[4] names a bf16 HardNet path: same keypoints, descriptors at bf16's own tolerance
        try:
            lafs_ref, cnt_ref = lafs.clone(), cnt.clone()       # run() returns the pipeline's own (reused) buffers
            hn.set_engine(L.ENGINE_TC2_BF16)
            l2, r2, d2, c2 = pipe.run(img.to(DEV))
            torch.cuda.synchronize()
            assert torch.equal(c2, cnt_ref) and torch.equal(l2[0, :n], lafs_ref[0, :n])
            rb = parity_report(oL, odesc, l2[0, :n].cpu(), d2[0, :n].cpu(), "4k, HardNet bf16 operands, vs oracle")
            assert rb["dd"] < 1e-2, rb
        finally:
            hn.set_engine(L.ENGINE_TC2)


def test_handcrafted_estimators_8f(L):
    """OrientationDetector / AffineShapeEstimator (SURVEY 8f): CUDA vs oracle on reference-extracted 19x19 patches, and the
    default detector (OriNet=None -> gradient-histogram orientation) end to end against the reference's golden output.  (The
    reference's own Baumberg LOOP raises TypeError under python3 - Utils.py:54 passes a stray dict - so only the module is pinned;
    ours additionally runs the 16-iteration loop of examples/hesaffnet/hesaffBaum.py:40.)"""
    from affnet_b200.HandCraftedModules import AffineShapeEstimator, OrientationDetector
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    z = gold("handcrafted.npz")
    P = torch.from_numpy(z["patches19"])
    ang = OrientationDetector(patch_size=19)(P.to(DEV)).cpu()
    ref = O.orientation_hist(P)
    agree = (torch.atan2(torch.sin(ang - ref), torch.cos(ang - ref)).abs() < 1e-5).float().mean().item()
    assert agree == 1.0, agree             # same patches -> same bins (r02 diagnostic scripts/ori_bins_diag.py: 200/200, no pixel changes its bin)
    A = AffineShapeEstimator(patch_size=19)(P.to(DEV)).cpu()
    assert (A - O.baumberg_shape(P)).abs().max() < 1e-4
    img = crop_img()
    det = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=300, border=5, num_Baum_iters=0)
    dL, r = det(img.to(DEV), do_ori=True)
    gL = torch.from_numpy(z["default_dLAFs"])
    ia, ib = match_keypoints(gL, dL.cpu(), tol_px=0.05)
    same = ((gL[ia] - dL.cpu()[ib]).abs().amax(dim=(1, 2)) < 1e-2).float().mean().item()
    print("\ndefault detector (histogram orientation): matched %d/%d, identical LAF %.3f" % (len(ia), gL.shape[0], same))
    assert len(ia) >= gL.shape[0] - 3 and same >= 0.97        # an orientation bin may flip at an fp32 near-tie
    det16 = ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=300, border=5, num_Baum_iters=16)
    dL16, r16 = det16(img.to(DEV), do_ori=True)
    assert 0 < dL16.shape[0] <= 300 and bool(torch.isfinite(dL16).all())


def test_snn_matcher_8f(L, nets):
    """distance_matrix_vector + SNN ratio test (SURVEY 8f row 3) on real descriptors of two views."""
    from affnet_b200.Losses import distance_matrix_vector, match_snn
    aff, ori, hn = nets
    g = torch.Generator().manual_seed(21)
    d1 = torch.nn.functional.normalize(torch.randn(700, 128, generator=g), dim=1)
    d2 = torch.cat([torch.nn.functional.normalize(d1[:400] + 0.25 * torch.randn(400, 128, generator=g), dim=1),
                    torch.nn.functional.normalize(torch.randn(333, 128, generator=g), dim=1)])
    D = distance_matrix_vector(d1.to(DEV), d2.to(DEV)).cpu()
    assert (D - O.distance_matrix_vector(d1, d2)).abs().max() < 1e-5
    i1, i2, mn, sec = match_snn(d1.to(DEV), d2.to(DEV), 0.8)
    o1, o2, omn, osec = O.match_snn(d1, d2, 0.8)
    assert (mn.cpu() - omn).abs().max() < 1e-5 and (sec.cpu() - osec).abs().max() < 1e-5
    assert torch.equal(i1.cpu(), o1) and torch.equal(i2.cpu(), o2)
    assert 0 < i1.numel() <= 700


def test_lafs2ell_t_8f(L, tmp_path):
    """8f row 4: LAFs2ellT on the device against the golden from the unmodified reference (fp32 closed-form SVD: 1e-5 relative),
    NaN for the degenerate row as in the reference, and the text writer."""
    from affnet_b200.LAF import LAFs2ellT, save_ells
    z = gold("ell.npz")
    g = torch.from_numpy(z["ell"])
    e = LAFs2ellT(torch.from_numpy(z["lafs"]).to(DEV)).cpu()
    assert torch.equal(torch.isnan(e), torch.isnan(g))
    ok = ~torch.isnan(g).any(dim=1)
    scale = g[ok][:, 2:].abs().max(dim=1, keepdim=True).values      # b is ~0 for near-circular regions: compare against the matrix scale
    err = ((e[ok][:, 2:] - g[ok][:, 2:]).abs() / scale).max(dim=1).values
    # the closed form takes the small singular value from sqrt((sum - dif) / 2): fp32 cancellation grows with the elongation^2 of
    # the region (the reference's own fp32 result is 2.7e-4 off its float64 value on the worst synthetic LAF here, elongation 308).
    # Detected regions have elongation < 6 (eigen-ratio filter); they get the tight bound, the degenerate synthetic ones a loose one.
    sv = torch.linalg.svdvals(torch.from_numpy(z["lafs"])[ok][:, :, :2].double())
    elong = sv[:, 0] / sv[:, 1]
    tight = elong < 6
    print("\nLAFs2ellT: max error (of the ellipse matrix scale) %.2e over %d regions with elongation < 6, %.2e over the %d others" % (
        err[tight].max().item(), int(tight.sum()), err[~tight].max().item(), int((~tight).sum())))
    assert torch.equal(e[ok][:, :2], g[ok][:, :2]) and err[tight].max() < 2e-5 and err[~tight].max() < 2e-2
    assert LAFs2ellT(torch.zeros(0, 2, 3, device=DEV)).shape == (0, 5)
    f = tmp_path / "ells.txt"
    save_ells(str(f), e[ok])
    back = np.loadtxt(str(f))
    assert back.shape == (int(ok.sum()), 5) and np.allclose(back, e[ok].numpy(), rtol=0, atol=1e-9 + 1e-7 * np.abs(e[ok].numpy()).max())


@pytest.mark.parametrize("mode", ["orinet", "noori", "hcori"])
def test_graf_1_to_6_application_counts(L, nets, mode):
    """The reference's own end-to-end check (train_AffNet_test_on_graffity.py:262-300) through the CUDA path: detect + describe graf
    img1 and img6 (K=3000), SNN matcher on the device, reprojection check by the oracle.  Counts of the unmodified reference:
    281/91 (hand-crafted orientation), 309/90 (OriNet), 104/18 (no orientation); a handful of the 6000 keypoints differ (eig-ratio
    filter at the 1e-3 level, DESIGN.md section 2), so the counts may move by a few."""
    from affnet_b200.Losses import match_snn
    from affnet_b200.SparseImgRepresenter import ScaleSpaceAffinePatchExtractor
    aff, ori, hn = nets
    z, f = gold("graf_match.npz"), gold("graf_full.npz")
    kw = dict(mrSize=5.192, num_features=3000, border=5, num_Baum_iters=1, AffNet=aff)
    if mode == "orinet":
        kw["OriNet"] = ori
    det = ScaleSpaceAffinePatchExtractor(**kw)
    out = []
    for rgb in (f["rgb"], z["rgb6"]):
        dL, _ = det(gray_from_rgb(rgb).to(DEV), do_ori=mode != "noori")
        out.append((dL, hn(det.extract_patches_from_pyr(dL, PS=32))))
    (L1, d1), (L2, d2) = out
    assert L1.size(0) == int(z[mode + "_n1"]) and L2.size(0) == int(z[mode + "_n2"])
    i1, i2, _, _ = match_snn(d1, d2, float(z["snn"]))
    _, keep, _ = O.gt_correspondences(L1[i1].cpu(), L2[i2].cpu(), torch.from_numpy(z["H1to6"]), float(z["px"]))
    tent, true = int(i1.numel()), int(keep.numel())
    print("\ngraf 1<->6 %s: %d tentatives / %d true (reference %d / %d)" % (mode, tent, true, int(z[mode + "_tent"]), int(z[mode + "_true"])))
    assert abs(tent - int(z[mode + "_tent"])) <= max(4, 0.03 * int(z[mode + "_tent"]))
    if mode != "hcori":
        assert abs(true - int(z[mode + "_true"])) <= max(4, 0.05 * int(z[mode + "_true"]))
        return
    # Hand-crafted orientation = arg-max over 36 histogram bins.  The kernel reproduces the reference's bins exactly on identical patches
    # (test_handcrafted_estimators_8f); end to end the separable blur's 3e-4 pyramid differences reach the 19x19 patches, and a keypoint
    # whose two best bins are a near-tie then takes the other bin (10 degrees or more away: a different descriptor, which is what moves
    # the loose "true" count).  Accounted for per keypoint: every keypoint whose orientation differs from the oracle's must be such a near-tie.
    assert abs(true - int(z[mode + "_true"])) <= max(6, 0.08 * int(z[mode + "_true"]))
    oL, _, st = O.detect(gray_from_rgb(f["rgb"]), W["affnet"], None, 3000, do_ori=True, debug=True)
    sm = O.orientation_hist_bins(st["debug"]["ori"]["patches"])
    top = sm.topk(2, dim=1).values
    margin = (top[:, 0] - top[:, 1]) / top[:, 0]
    ia, ib = match_keypoints(oL, L1.cpu())
    eA = ((oL[ia][:, :, :2] - L1.cpu()[ib][:, :, :2]).abs().amax(dim=(1, 2)) / (oL[ia][:, 0, 0] * oL[ia][:, 1, 1] - oL[ia][:, 0, 1] * oL[ia][:, 1, 0]).abs().sqrt())
    flipped = (eA > 1e-2).nonzero().view(-1)
    print("img1: %d of %d matched keypoints take another orientation bin than the oracle; their top-2 bin margins (oracle): %s" % (
        flipped.numel(), len(ia), ["%.1e" % margin[ia[i]].item() for i in flipped.tolist()]))
    assert len(ia) >= 0.995 * oL.shape[0] and flipped.numel() <= 0.005 * len(ia)
    # ... or (tests/helpers.py::orientation_boundary_shares) own a pixel on a histogram-bin boundary that outweighs its bin margin: the reference
    # adds a pixel's whole weight to the LOWER bin only, so such a pixel changes bins under any perturbation
    _, share = orientation_boundary_shares(st["debug"]["ori"]["patches"])
    assert all(margin[ia[i]].item() < 5e-3 or share[ia[i]].item() > margin[ia[i]].item() for i in flipped.tolist())
