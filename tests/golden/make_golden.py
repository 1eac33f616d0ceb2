"""Generates the golden fixtures in this directory by running the UNMODIFIED reference
(/root/reference, ducha-aiki/affnet @ da7cf51) on CPU in the build container.

    python tests/golden/make_golden.py

The reference pins no results of its own (no tests, no golden vectors - SURVEY.md §4), so these
files are what pins `oracle/affnet_oracle.py` to the reference.  Re-run only when the reference
changes.  Outputs (all .npz, compressed):

  weights.npz        state dicts of pretrained/AffNet.pth, pretrained/OriNet.pth, HardNet++.pth
  graf_crop.npz      256x320 crop of test-graf/img1.png, K=300: per-stage intermediates
  graf_full.npz      full test-graf/img1.png 800x640, K=2000, do_ori in {False, True}: final outputs
  nms_q4.npz         NMS3dAndComposeA on synthetic response maps with a non-trivial octave map (Q4)
  face_patches.npz   first 64 patches of examples/just_shape/img/face.png -> AffNetFast matrices
  nets_random.npz    the three nets on 32 random patches (input + outputs)
  handcrafted.npz    OrientationDetector / AffineShapeEstimator on 19x19 patches; default detector (OriNet=None) end to end
  ell.npz            LAFs2ellT (the Oxford-affine output of hesaffBaum.py) on the graf crop's final LAFs + synthetic LAFs
                     (`python tests/golden/make_golden.py ell` regenerates only this file from graf_crop.npz)
  graf_match.npz     the reference's own application test (train_AffNet_test_on_graffity.py:262-300): graf img1 <-> img6, K=3000,
                     HardNet + SNN 0.8 + 6 px reprojection check, for hand-crafted orientation / OriNet / no orientation:
                     tentative and true match counts, img6 and H1to6p (`... make_golden.py match`)
  distance.npz       Losses.distance_matrix_vector on seeded random descriptors (`... make_golden.py distance`)
"""
import contextlib
import io
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import ref_harness as R  # noqa: E402

warnings.filterwarnings("ignore")
torch.set_num_threads(8)


def quiet():
    return contextlib.redirect_stdout(io.StringIO())


def save(name, **kw):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **{k: (v.detach().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in kw.items()})
    print(name, "%.1f KB" % (os.path.getsize(path) / 1024.0))


def rgb_of(path):
    from PIL import Image
    return np.array(Image.open(path).convert("RGB"))


def gray_of(rgb):
    return torch.from_numpy(np.mean(rgb, axis=2).astype(np.float32)).view(1, 1, rgb.shape[0], rgb.shape[1])


def main():
    m = R.ref_modules()
    aff, ori, hn = R.load_nets()
    w = {}
    for pre, net in (("affnet", aff), ("orinet", ori), ("hardnet", hn)):
        for k, v in net.state_dict().items():
            if "num_batches_tracked" not in k:
                w[pre + "/" + k] = v
    save("weights.npz", **w)

    # ---------------- graf crop, per-stage --------------------------------------------------
    rgb = rgb_of(R.REF + "/test-graf/img1.png")
    crop = np.ascontiguousarray(rgb[100:356, 200:520])
    img = gray_of(crop)
    K = 300
    out = dict(rgb=crop, K=K)
    det = R.make_detector(aff, ori, num_features=K)
    with torch.no_grad(), quiet():
        resp, LAFs, pidx, lidx = det.multiScaleDetector(img, int(1.5 * K))
        pyr = det.scale_pyr
        out["n_oct"] = len(pyr)
        for o in range(len(pyr)):
            for l in range(5):
                out["pyr_sum_%d_%d" % (o, l)] = pyr[o][l].double().sum()
        out["pyr_1_2"] = pyr[1][2][0, 0]
        out["pyr_0_4_rows"] = pyr[0][4][0, 0, 100:108]
        out["hess_1_2"] = det.RespNet(pyr[1][2], det.sigmas[1][2])[0, 0]
        out.update(det_resp=resp, det_LAFs=LAFs, det_pidx=pidx, det_lidx=lidx)
        L2 = LAFs.clone()
        L2[:, 0:2, 0:2] = det.mrSize * L2[:, :, 0:2]
        inv = m["LAF"].get_inverted_pyr_index(pyr, pidx, lidx)
        P = m["LAF"].extract_patches_from_pyramid_with_inv_index(pyr, inv, L2, PS=32)
        A = m["Utils"].batched_forward(aff, P, 256)
        out.update(aff_patches=P[:64], aff_A=A)
        r2, L3, p2, l2 = det.getAffineShape(resp, L2, pidx, lidx, K)
        out.update(shape_resp=r2, shape_LAFs=L3, shape_pidx=p2, shape_lidx=l2)
        inv = m["LAF"].get_inverted_pyr_index(pyr, p2, l2)
        P = m["LAF"].extract_patches_from_pyramid_with_inv_index(pyr, inv, L3, PS=32)
        Rm = ori(P)
        out.update(ori_patches=P[:64], ori_R=Rm)
        for do_ori in (False, True):
            d = R.make_detector(aff, ori, num_features=K)
            dL, rr, pp, dd = R.run_full(d, hn, img, do_ori)
            o_, l_ = m["LAF"].get_pyramid_and_level_index_for_LAFs(dL, d.sigmas, d.pix_dists, 32)
            tag = "ori" if do_ori else "noori"
            out.update({tag + "_dLAFs": dL, tag + "_resp": rr, tag + "_desc_patches": pp[:64], tag + "_desc": dd,
                        tag + "_desc_oct": o_, tag + "_desc_lvl": l_})
    save("graf_crop.npz", **out)

    # ---------------- graf full, final outputs only ----------------------------------------
    img = gray_of(rgb)
    out = dict(rgb=rgb, K=2000)
    for do_ori in (False, True):
        d = R.make_detector(aff, ori, num_features=2000)
        dL, rr, pp, dd = R.run_full(d, hn, img, do_ori)
        tag = "ori" if do_ori else "noori"
        out.update({tag + "_dLAFs": dL, tag + "_resp": rr, tag + "_desc": dd.half()})
    with torch.no_grad(), quiet():
        rall, _, pa, la = d.multiScaleDetector(img, -1)
    out["cand_counts"] = np.array([[int(((pa == o) & (la == l)).sum()) for l in range(3)] for o in range(len(d.scale_pyr))])
    save("graf_full.npz", **out)

    # ---------------- NMS with octave map (Q4) ---------------------------------------------
    g = torch.Generator().manual_seed(7)
    h, wd = 40, 56
    base = torch.rand(1, 1, h, wd, generator=g)
    import torch.nn.functional as F
    maps = []
    for i in range(3):
        x = torch.rand(1, 1, h, wd, generator=g) * 400.0
        x = F.avg_pool2d(F.pad(x, (1, 1, 1, 1), "replicate"), 3, stride=1)
        maps.append(x.contiguous())
    omap = (torch.rand(h, wd, generator=g) * 4.3).byte().view(1, 1, h, wd)  # values 0..4
    omap[0, 0, :, : wd // 2] = 0
    scales = [1.6, 2.0158736798317967, 2.5398416831491195]
    out = dict(low=maps[0][0, 0], cur=maps[1][0, 0], high=maps[2][0, 0], omap=omap[0, 0], scales=np.array(scales))
    for nf, tag in ((0, "all"), (20, "top20")):
        nms = m["HandCraftedModules"].NMS3dAndComposeA(w=wd, h=h, border=5, mrSize=5.192)
        with torch.no_grad():
            r, A, om2 = nms(maps[0].clone(), maps[1].clone(), maps[2].clone(), num_features=nf, octaveMap=omap.clone(), scales=scales)
        out.update({tag + "_resp": r, tag + "_LAFs": A, tag + "_omap": om2[0, 0]})
    save("nms_q4.npz", **out)

    # ---------------- just_shape: face patches -> AffNet ----------------------------------
    import cv2
    face = cv2.imread(R.REF + "/examples/just_shape/img/face.png", 0)
    wdt = face.shape[1]
    pts = np.stack([cv2.resize(face[i * wdt:(i + 1) * wdt], (32, 32), interpolation=cv2.INTER_LINEAR) for i in range(64)])
    P = torch.from_numpy(pts.astype(np.float32) / 255.0).view(64, 1, 32, 32)
    with torch.no_grad():
        A = aff(P)
    save("face_patches.npz", patches_u8=pts, A=A)

    # ---------------- hand-crafted estimators (SURVEY 8f rows 1-2) ---------------------------
    import torch.nn.functional as F2  # noqa: F401
    crop_img = gray_of(crop)
    # NB: the reference's own Baumberg loop (AffNet=None, num_Baum_iters > 0) raises TypeError under python3 because
    # batched_forward passes a stray dict to AffineShapeEstimator.forward (Utils.py:54,66); only the module itself is runnable.
    det0 = m["SparseImgRepresenter"].ScaleSpaceAffinePatchExtractor(mrSize=5.192, num_features=300, border=5, num_Baum_iters=0)
    with torch.no_grad(), quiet():
        dL0, r0 = det0(crop_img, do_ori=True)       # detector + gradient-histogram orientation (OriNet=None default)
        resp, LAFs, pidx, lidx = det0.multiScaleDetector(crop_img, 450)
        L2 = LAFs.clone(); L2[:, 0:2, 0:2] = det0.mrSize * L2[:, :, 0:2]
        inv = m["LAF"].get_inverted_pyr_index(det0.scale_pyr, pidx, lidx)
        P19 = m["LAF"].extract_patches_from_pyramid_with_inv_index(det0.scale_pyr, inv, L2, PS=19)
        od = m["HandCraftedModules"].OrientationDetector(patch_size=19)
        ae = m["HandCraftedModules"].AffineShapeEstimator(patch_size=19)
        save("handcrafted.npz", patches19=P19[:200], angle=od(P19[:200]), A=ae(P19[:200]), default_dLAFs=dL0, default_resp=r0)

    # ---------------- nets on random patches ----------------------------------------------
    P = torch.rand(32, 1, 32, 32, generator=g) * 255.0
    with torch.no_grad():
        save("nets_random.npz", patches=P, affnet_A=aff(P), orinet_R=ori(P), orinet_angle=ori(P, return_rot_matrix=False),
             hardnet_desc=hn(P))


def make_ell():
    m = R.ref_modules()
    z = np.load(os.path.join(HERE, "graf_crop.npz"))
    g = torch.Generator().manual_seed(11)
    A = torch.randn(64, 2, 2, generator=g) * 6.0
    A[:, 0, 0] = A[:, 0, 0].abs() + 4.0; A[:, 1, 1] = A[:, 1, 1].abs() + 4.0       # positive determinant
    syn = torch.cat([A, torch.rand(64, 2, 1, generator=g) * 300.0], dim=2)
    lafs = torch.cat([torch.from_numpy(z["ori_dLAFs"]), torch.from_numpy(z["noori_dLAFs"]), syn]).float()
    with torch.no_grad():
        ell = m["LAF"].LAFs2ellT(lafs)
    # host-side output format (LAF.py:225-240, numpy float64 SVD) on the rows it is defined for (positive determinant)
    ln = lafs.numpy()
    pos = (ln[:, 0, 0] * ln[:, 1, 1] - ln[:, 0, 1] * ln[:, 1, 0]) > 0
    ell_host = m["LAF"].LAFs2ell(ln[pos])
    save("ell.npz", lafs=lafs, ell=ell, host_rows=np.nonzero(pos)[0], ell_host=ell_host)


def make_jit():
    """f4: the TorchScript exports of the reference (convertJIT/*.pt) run on CPU: raw head outputs on real and random patches."""
    z = np.load(os.path.join(HERE, "graf_crop.npz"))
    g = torch.Generator().manual_seed(17)
    P = torch.cat([torch.from_numpy(z["aff_patches"])[:96], torch.rand(32, 1, 32, 32, generator=g) * 255.0]).float()
    aff = torch.jit.load(os.path.join(R.REF, "convertJIT", "AffNetJIT.pt"), map_location="cpu").eval()
    ori = torch.jit.load(os.path.join(R.REF, "convertJIT", "OriNetJIT.pt"), map_location="cpu").eval()
    with torch.no_grad():
        save("jit.npz", patches=P, affnet_raw=aff(P), orinet_raw=ori(P))


def make_match():
    import importlib
    m = R.ref_modules()
    RS, LS = importlib.import_module("ReprojectionStuff"), importlib.import_module("Losses")
    aff, ori, hn = R.load_nets()
    rgb1, rgb6 = rgb_of(R.REF + "/test-graf/img1.png"), rgb_of(R.REF + "/test-graf/img6.png")
    H = np.loadtxt(R.REF + "/test-graf/H1to6p")
    out = dict(rgb6=rgb6, H1to6=H, K=3000, snn=0.8, px=6.0)
    for mode in ("hcori", "orinet", "noori"):
        det = R.make_detector(aff, ori if mode == "orinet" else None, num_features=3000)
        L1, _, _, d1 = R.run_full(det, hn, gray_of(rgb1), mode != "noori")
        L2, _, _, d2 = R.run_full(det, hn, gray_of(rgb6), mode != "noori")
        with torch.no_grad():                                       # train_AffNet_test_on_graffity.py:289-300
            dm = LS.distance_matrix_vector(d1, d2)
            mn, i2 = torch.min(dm, 1)
            dm[:, i2] = 100000
            sec, _ = torch.min(dm, 1)
            mask = (mn / (sec + 1e-8)) <= 0.8
            t1, t2 = torch.arange(0, i2.size(0))[mask].long(), i2[mask].long()
            _, pi1, _ = RS.get_GT_correspondence_indexes(L1[t1], L2[t2], torch.from_numpy(H).float(), dist_threshold=6)
        out.update({mode + "_n1": L1.size(0), mode + "_n2": L2.size(0), mode + "_tent": t1.numel(), mode + "_true": pi1.numel(),
                    mode + "_t1": t1, mode + "_t2": t2})
        print(mode, L1.size(0), L2.size(0), t1.numel(), "tentatives", pi1.numel(), "true")
    save("graf_match.npz", **out)


def make_distance():
    """8f row 3: Losses.distance_matrix_vector on 50 x 70 seeded random descriptors (inputs stored with the output)."""
    import importlib
    R.ref_modules()
    LS = importlib.import_module("Losses")
    g = torch.Generator().manual_seed(5)
    a, b = torch.randn(50, 128, generator=g), torch.randn(70, 128, generator=g)
    with torch.no_grad():
        save("distance.npz", a=a, b=b, d=LS.distance_matrix_vector(a, b))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "ell":
        make_ell()
    elif len(sys.argv) > 1 and sys.argv[1] == "match":
        make_match()
    elif len(sys.argv) > 1 and sys.argv[1] == "jit":
        make_jit()
    elif len(sys.argv) > 1 and sys.argv[1] == "distance":
        make_distance()
    else:
        main()
        make_ell()
        make_match()
        make_jit()
        make_distance()
