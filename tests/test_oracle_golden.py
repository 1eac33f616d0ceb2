"""CPU tests: pin oracle/affnet_oracle.py against golden vectors produced by the unmodified
reference (tests/golden/make_golden.py).  Tolerances are stated per stage."""
import numpy as np
import pytest
import torch

import affnet_oracle as O
from helpers import gold, load_weights, gray_from_rgb, match_keypoints

W = load_weights()


def T(a):
    return torch.from_numpy(np.asarray(a))


def test_gauss_kernel_sizes_q1():
    # SURVEY §8a Q1: sigma -> (k, pad)
    for s, k in ((1.5199, 11), (1.2263, 9), (1.5450, 11), (1.9466, 13), (2.4525, 15)):
        assert O.gauss_kernel_size(s) == k
    g = O.gauss_kernel_1d(1.2263)
    assert abs(np.outer(g, g) - O.gauss_kernel_2d(1.2263)).max() < 1e-16   # separable to f64 rounding


def test_pyramid_plan_graf():
    sizes, bs, sig, pix = O.pyramid_plan(640, 800)
    assert sizes == [(640, 800), (320, 400), (160, 200), (80, 100), (40, 50), (20, 25)]
    assert sig[0][3] == 3.1999999999999997 and pix[3] == [8.0] * 5
    assert abs(bs[0][0] - 1.5198684) < 1e-6 and [O.gauss_kernel_size(s) for s in bs[0][1:]] == [9, 11, 13, 15]


def test_detector_stage_bit_exact_vs_reference_golden():
    z = gold("graf_crop.npz")
    img = gray_from_rgb(z["rgb"])
    K = int(z["K"])
    pyr, sig, pix = O.scale_pyramid(img)
    assert len(pyr) == int(z["n_oct"])
    for o in range(len(pyr)):
        for l in range(5):
            assert abs(pyr[o][l].double().sum().item() - float(z["pyr_sum_%d_%d" % (o, l)])) < 1e-6
    assert torch.equal(pyr[1][2][0, 0], T(z["pyr_1_2"]))          # same torch op => bit exact
    assert torch.equal(pyr[0][4][0, 0, 100:108], T(z["pyr_0_4_rows"]))
    assert torch.equal(O.hessian_response(pyr[1][2], sig[1][2])[0, 0], T(z["hess_1_2"]))
    resp, LAFs, pidx, lidx = O.multi_scale_detector(pyr, sig, int(1.5 * K), 5.192)
    assert torch.equal(resp, T(z["det_resp"]))                     # identical index set and order
    assert torch.equal(pidx, T(z["det_pidx"])) and torch.equal(lidx, T(z["det_lidx"]))
    assert (LAFs - T(z["det_LAFs"])).abs().max() < 1e-6            # soft-argmax conv order: 6e-8


def test_nms_octave_map_q4():
    z = gold("nms_q4.npz")
    low, cur, high = (T(z[k]).view(1, 1, *z[k].shape) for k in ("low", "cur", "high"))
    for nf, tag in ((0, "all"), (20, "top20")):
        r, A, om, idxs = O.nms3d_and_compose(low, cur, high, nf, z["omap"].copy(), list(z["scales"]), 5.192)
        assert torch.equal(r, T(z[tag + "_resp"]))
        assert (r < 0).any() or nf > 0                             # Q4: re-detected pixels go negative
        assert np.array_equal(om, z[tag + "_omap"])                # uint8 wrap reproduced
        assert (A - T(z[tag + "_LAFs"])).abs().max() < 1e-6


def test_sampler_and_affnet_stage():
    z = gold("graf_crop.npz")
    img = gray_from_rgb(z["rgb"])
    pyr, sig, pix = O.scale_pyramid(img)
    L = T(z["det_LAFs"]).clone()
    L[:, 0:2, 0:2] = 5.192 * L[:, :, 0:2]
    P = O.extract_patches_from_pyramid(pyr, T(z["det_pidx"]), T(z["det_lidx"]), L, 32)
    # closed-form f64 bilinear vs torch's fp32 affine_grid+grid_sample: coordinate rounding x gradient
    assert (P[:64] - T(z["aff_patches"])).abs().max() < 2e-2      # on a 0..255 scale
    A = O.affnet_forward(T(z["aff_patches"]), W["affnet"])
    assert (A - T(z["aff_A"])[:64]).abs().max() < 1e-5
    A_all = O.affnet_forward(P, W["affnet"])
    assert (A_all - T(z["aff_A"])).abs().max() < 1e-3


def test_shape_filter_given_reference_A():
    z = gold("graf_crop.npz")
    K = int(z["K"])
    L = T(z["det_LAFs"]).clone(); L[:, 0:2, 0:2] = 5.192 * L[:, :, 0:2]
    A = T(z["aff_A"])
    newL = torch.cat([torch.bmm(A, L[:, :, :2]), L[:, :, 2:]], 2)
    mask = O.shape_filter_mask(A, newL)
    resp = T(z["det_resp"])
    if int(mask.sum()) > K:
        r, idxs = torch.topk(resp * mask.float(), k=K)
    else:
        idxs = mask.nonzero().view(-1); r = resp[idxs]
    assert torch.equal(r, T(z["shape_resp"]))                      # identical selection given identical A
    assert (newL[idxs] - T(z["shape_LAFs"])).abs().max() < 1e-6


def test_orinet_and_hardnet_stage():
    z = gold("graf_crop.npz")
    R = O.orinet_forward(T(z["ori_patches"]), W["orinet"])
    assert (R - T(z["ori_R"])[:64]).abs().max() < 1e-5
    d = O.hardnet_forward(T(z["ori_desc_patches"]), W["hardnet"])
    assert (d - T(z["ori_desc"])[:64]).abs().max() < 1e-5


def test_level_selection_a15():
    z = gold("graf_crop.npz")
    sizes, bs, sig, pix = O.pyramid_plan(*z["rgb"].shape[:2])
    for tag in ("noori", "ori"):
        o, l = O.pyramid_level_for_lafs(T(z[tag + "_dLAFs"]), sig, pix, 32)
        assert np.array_equal(o.numpy(), z[tag + "_desc_oct"]) and np.array_equal(l.numpy(), z[tag + "_desc_lvl"])


def test_nets_on_random_patches_and_face():
    z = gold("nets_random.npz")
    P = T(z["patches"])
    assert (O.affnet_forward(P, W["affnet"]) - T(z["affnet_A"])).abs().max() < 1e-5
    assert (O.orinet_forward(P, W["orinet"]) - T(z["orinet_R"])).abs().max() < 1e-5
    assert (O.orinet_angle(P, W["orinet"]) - T(z["orinet_angle"])).abs().max() < 1e-5
    assert (O.hardnet_forward(P, W["hardnet"]) - T(z["hardnet_desc"])).abs().max() < 1e-5
    f = gold("face_patches.npz")
    P = torch.from_numpy(f["patches_u8"].astype(np.float32) / 255.0).view(-1, 1, 32, 32)
    A = O.affnet_forward(P, W["affnet"])
    assert (A - T(f["A"])).abs().max() < 1e-5
    # SURVEY §8c known answers
    assert abs(A[0, 0, 0] - 0.9761) < 1e-4 and abs(A[0, 1, 0] - 0.0652) < 1e-4 and abs(A[1, 1, 0] - 0.2110) < 1e-4


@pytest.mark.parametrize("do_ori", [False, True])
def test_end_to_end_crop(do_ori):
    z = gold("graf_crop.npz")
    img = gray_from_rgb(z["rgb"])
    tag = "ori" if do_ori else "noori"
    dL, resp, st = O.detect(img, W["affnet"], W["orinet"], int(z["K"]), do_ori=do_ori)
    desc, _, _ = O.describe(dL, st, W["hardnet"])
    gL, gd = T(z[tag + "_dLAFs"]), T(z[tag + "_desc"])
    ia, ib = match_keypoints(gL, dL)
    assert len(ia) >= 0.995 * gL.shape[0]                          # SURVEY §8a Q7(ii)
    assert (gL[ia] - dL[ib]).abs().max() < 2e-2                    # px units; fp32 sampler noise -> AffNet/OriNet
    assert (gd[ia] - desc[ib]).abs().max() < 5e-3


def test_end_to_end_graf_full_known_answers():
    z = gold("graf_full.npz")
    img = gray_from_rgb(z["rgb"])
    dL, resp, st = O.detect(img, W["affnet"], None, 2000, do_ori=False)
    gL = T(z["noori_dLAFs"])
    # SURVEY §8c: first LAFs of graf img1
    assert (gL[0] - torch.tensor([[16.8363, 0, 467.4685], [0.8120, 17.7178, 264.4630]])).abs().max() < 1e-3
    ia, ib = match_keypoints(gL, dL)
    assert len(ia) >= 0.995 * 2000
    assert (gL[ia] - dL[ib]).abs().max() < 2e-2
    desc, _, _ = O.describe(dL, st, W["hardnet"])
    assert (T(z["noori_desc"]).float()[ia] - desc[ib]).abs().max() < 5e-3
    # candidate counts per (octave, level): 7885 in total (SURVEY §8c)
    assert int(z["cand_counts"].sum()) == 7885


def test_handcrafted_estimators_8f():
    """SURVEY 8(f) rows 1-2: gradient-histogram orientation and the Baumberg step against the reference's outputs."""
    z = gold("handcrafted.npz")
    P = T(z["patches19"])
    assert torch.equal(O.orientation_hist(P), T(z["angle"]))
    assert (O.baumberg_shape(P) - T(z["A"])).abs().max() < 1e-6


def test_orientation_histogram_has_bin_boundary_discontinuities():
    """The accounting of the GPU application test (test_gpu_parity.py::test_graf_1_to_6_application_counts[hcori]) rests on this property of the
    reference's gradient histogram: only the lower-bin weight of a pixel is accumulated, so a pixel ON a bin boundary switches bins under an
    epsilon change.  (i) Constructed: a ramp patch whose gradient direction moves across a bin boundary by 2e-4 bins changes its histogram's mass 18x; (ii) in the graf img1 keypoints such pixels exist (helpers.orientation_boundary_shares finds a keypoint whose
    boundary pixel outweighs its bin margin)."""
    import math

    from helpers import orientation_boundary_shares
    # (i) a linear ramp: every interior pixel has the same gradient direction, 1e-4 bins below / above the boundary between bins 19 and 20
    PS = 19
    yy, xx = torch.meshgrid(torch.arange(PS, dtype=torch.float64), torch.arange(PS, dtype=torch.float64), indexing="ij")
    hists = []
    for eps in (-1e-4, 1e-4):
        th = (2.0 * math.pi) * (20.0 + eps) / 36.0 - math.pi          # o_big = 20 +- 1e-4 bins
        ramp = (-(xx * math.cos(th) + yy * math.sin(th)) * 3.0).float().view(1, 1, PS, PS)   # gx = 0.5 x[j-1] - 0.5 x[j+1] = 3 cos(th), gy = 3 sin(th)
        hists.append(O.orientation_hist_bins(ramp)[0])
    # below the boundary the interior's weight lands in bin 19 scaled by (1 - 0.9999); above it bin 20 takes all of it: the histogram's
    # mass jumps 18x for a change of direction of 2e-4 bins
    # (what is left below the boundary are the border pixels, whose replicate-padded gradients point elsewhere)
    assert hists[1][20] > 10 * hists[0][20] and hists[1].sum() > 10 * hists[0].sum(), (hists[0], hists[1])
    # (ii) graf img1, K = 3000 with hand-crafted orientation
    f = gold("graf_full.npz")
    _, _, st = O.detect(gray_from_rgb(f["rgb"]), W["affnet"], None, 3000, do_ori=True, debug=True)
    margin, share = orientation_boundary_shares(st["debug"]["ori"]["patches"])
    risky = ((share > margin) & (margin > 1e-2)).nonzero().view(-1)
    assert margin.shape == (st["debug"]["ori"]["patches"].size(0),) and risky.numel() >= 1, risky


def test_distance_matrix_vs_reference_golden():
    """Losses.distance_matrix_vector (SURVEY 8f row 3) against the reference's output on the same seeded inputs
    (tests/golden/make_golden.py::make_distance)."""
    z = gold("distance.npz")
    assert torch.equal(O.distance_matrix_vector(T(z["a"]), T(z["b"])), T(z["d"]))


def test_lafs2ell_t_matches_reference_bit_exactly():
    """8f row 4: the Oxford-affine output format.  One synthetic LAF has a negative determinant: NaN, as in the reference."""
    z = gold("ell.npz")
    e = O.lafs_to_ell_t(torch.from_numpy(z["lafs"]))
    g = torch.from_numpy(z["ell"])
    assert torch.equal(torch.isnan(e), torch.isnan(g)) and int(torch.isnan(g).any(dim=1).sum()) == 1
    ok = ~torch.isnan(g).any(dim=1)
    assert torch.equal(e[ok], g[ok])
    assert O.lafs_to_ell_t(torch.zeros(0, 2, 3)).shape == (0, 5)


@pytest.mark.parametrize("mode", ["orinet", "noori", "hcori"])
def test_graf_1_to_6_application_counts(mode):
    """The reference's own end-to-end check (train_AffNet_test_on_graffity.py:262-300): graf img1 <-> img6, K=3000, HardNet, SNN 0.8,
    6 px reprojection: tentatives / true matches of the unmodified reference (281/91 hand-crafted orientation, 309/90 OriNet,
    104/18 none) from the oracle restatement.  The gradient-histogram orientation flips one arg-max bin in 6000 keypoints."""
    z, f = gold("graf_match.npz"), gold("graf_full.npz")
    x1, x6 = gray_from_rgb(f["rgb"]), gray_from_rgb(z["rgb6"])
    ori = W["orinet"] if mode == "orinet" else None
    L1, _, d1 = O.detect_and_describe(x1, W["affnet"], ori, W["hardnet"], num_features=3000, do_ori=mode != "noori")
    L2, _, d2 = O.detect_and_describe(x6, W["affnet"], ori, W["hardnet"], num_features=3000, do_ori=mode != "noori")
    tent, true = O.match_and_verify(L1, d1, L2, d2, torch.from_numpy(z["H1to6"]), float(z["snn"]), float(z["px"]))
    slack = 2 if mode == "hcori" else 0
    assert abs(tent - int(z[mode + "_tent"])) <= slack and abs(true - int(z[mode + "_true"])) <= slack, (tent, true)


def test_raw_heads_match_the_reference_torchscript_exports():
    """f4: convertJIT/AffNetJIT.pt returns xy + [1, 0, 1], OriNetJIT.pt the mean of tanh over the 3x3 map (golden: the .pt files run on CPU)."""
    z = gold("jit.npz")
    P = torch.from_numpy(z["patches"])
    a = O.affnet_raw(P, W["affnet"]) + torch.tensor([[1.0, 0.0, 1.0]])
    assert (a - torch.from_numpy(z["affnet_raw"])).abs().max() < 1e-5
    assert (O.orinet_raw(P, W["orinet"]) - torch.from_numpy(z["orinet_raw"])).abs().max() < 1e-5
