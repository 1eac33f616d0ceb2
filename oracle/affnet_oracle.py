"""CPU oracle for the HesAffNet + HardNet detect-and-describe hot path.

TEST INFRASTRUCTURE, NOT PRODUCT.  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s
`cpu_baseline` / `--impl reference` legs may import this module.  The product (`affnet_b200/`)
never does; it fails loudly when its CUDA library is missing.

This is an independent restatement (plain PyTorch-CPU / numpy, fp32 unless noted) of the algorithm
the reference (ducha-aiki/affnet @ da7cf51) executes under Python 3 / torch 2.x.  Every function
cites the reference file:line it follows.  Parity is PINNED: `tests/golden/make_golden.py` ran the
unmodified reference in the build container and committed its outputs under `tests/golden/`;
`tests/test_oracle_golden.py` checks this oracle against them.

Quirks reproduced on purpose (SURVEY.md §8a Q1-Q8): non-integer Gaussian tap spacing (Q1), the
+0.5 px soft-argmax bias (Q2), uint8 wrap of the octave map (Q4), mixed units in the boundary
check (Q5), per-octave normalisation by ceil-halved sizes (Q6).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------------------------
# a1  Gaussian blur                                            Utils.py:92-114, 150-166
# ----------------------------------------------------------------------------------------------


def gauss_kernel_size(sigma):
    """Utils.py:95-97: k = int(6 sigma + 1), forced odd."""
    k = int(2.0 * 3.0 * sigma + 1.0)
    if k % 2 == 0:
        k += 1
    return k


def gauss_kernel_1d(sigma):
    """Normalised 1-D factor g of the reference's 2-D kernel (float64).

    Utils.py:98-113: taps at linspace(-k/2, k/2, k) (py3 true division => spacing k/(k-1), Q1),
    w2d = exp(-(x^2+y^2)/(2 sigma^2)) / sum  ==  outer(g, g) with g = e/sum(e).
    """
    k = gauss_kernel_size(sigma)
    half = k / 2
    x = np.linspace(-half, half, k)
    e = np.exp(-(x * x) / (2.0 * sigma * sigma))
    return e / e.sum()


def gauss_kernel_2d(sigma):
    """The reference's dense kernel exactly as built (Utils.py:92-114), float64 [k,k]."""
    k = gauss_kernel_size(sigma)
    half = k / 2
    x = np.linspace(-half, half, k)
    xv, yv = np.meshgrid(x, x, sparse=False, indexing="xy")
    ker = np.exp(-((xv ** 2 + yv ** 2) / (2.0 * sigma * sigma)))
    return ker / np.sum(ker)


def gaussian_blur(x, sigma):
    """Utils.py:160-166: replicate pad floor(k/2), dense k x k cross-correlation, fp32."""
    ker = gauss_kernel_2d(sigma)
    k = ker.shape[0]
    pad = int(np.floor(float(k) / 2.0))
    w = torch.from_numpy(ker.astype(np.float32)).view(1, 1, k, k)
    return F.conv2d(F.pad(x, (pad, pad, pad, pad), "replicate"), w, padding=0)


# ----------------------------------------------------------------------------------------------
# a2  Scale pyramid                                           HandCraftedModules.py:13-56
# ----------------------------------------------------------------------------------------------


def pyramid_plan(H, W, nlevels=3, init_sigma=1.6, border=5):
    """Sizes/sigmas of the pyramid without computing it (host logic shared by tests).

    Returns (sizes[o]=(h,w), blur_sigmas[o][l] (sigma of the blur that PRODUCES level l; level 0 of
    octave>0 is a decimation -> None), sigmas[o][l], pix_dists[o][l]).
    HandCraftedModules.py:23-56.  Python-float / numpy-float64 arithmetic as in the reference.
    """
    sigma_step = 2 ** (1.0 / float(nlevels))
    min_size = 2 * border + 2 + 1
    cur_sigma = 0.5
    sizes, blur_sigmas, sigmas, pix = [], [], [], []
    if init_sigma > cur_sigma:
        first = float(np.sqrt(init_sigma ** 2 - cur_sigma ** 2))
        cur_sigma = init_sigma
    else:
        first = None
    h, w = H, W
    pd = 1.0
    sizes.append((h, w)); blur_sigmas.append([first]); sigmas.append([cur_sigma]); pix.append([1.0])
    while True:
        for i in range(1, nlevels + 2):
            s = cur_sigma * np.sqrt(sigma_step * sigma_step - 1.0)
            blur_sigmas[-1].append(float(s))
            cur_sigma = cur_sigma * sigma_step
            sigmas[-1].append(cur_sigma)
            pix[-1].append(pd)
        pd = pd * 2.0
        cur_sigma = init_sigma
        nh, nw = (h + 1) // 2, (w + 1) // 2  # avg_pool2d(k=1, s=2): floor((h-1)/2)+1
        if nh <= min_size or nw <= min_size:
            break
        h, w = nh, nw
        sizes.append((h, w)); blur_sigmas.append([None]); sigmas.append([cur_sigma]); pix.append([pd])
    return sizes, blur_sigmas, sigmas, pix


def scale_pyramid(x, nlevels=3, init_sigma=1.6, border=5):
    """HandCraftedModules.py:23-56.  x: float32 [1,1,H,W].  Returns (pyr, sigmas, pix_dists)."""
    sizes, blur_sigmas, sigmas, pix = pyramid_plan(x.size(2), x.size(3), nlevels, init_sigma, border)
    pyr = []
    for o in range(len(sizes)):
        if o == 0:
            cur = gaussian_blur(x, blur_sigmas[0][0]) if blur_sigmas[0][0] is not None else x
        else:
            cur = pyr[o - 1][nlevels][:, :, ::2, ::2].contiguous()  # F.avg_pool2d(k=1, stride=2)
        levels = [cur]
        for l in range(1, nlevels + 2):
            cur = gaussian_blur(cur, blur_sigmas[o][l])
            levels.append(cur)
        pyr.append(levels)
        assert tuple(levels[0].shape[2:]) == sizes[o]
    return pyr, sigmas, pix


# ----------------------------------------------------------------------------------------------
# a3  Hessian response                                       HandCraftedModules.py:58-78
# ----------------------------------------------------------------------------------------------


def hessian_response(x, sigma):
    """abs(gxx*gyy - gxy^2) * sigma^4 with replicate (clamped) borders; x float32 [1,1,h,w].

    gxx = x[j-1] - 2x[j] + x[j+1]; gyy likewise vertically; gxy = two chained (0.5,0,-0.5)
    cross-correlations = 0.25*(x[i-1,j-1] - x[i-1,j+1] - x[i+1,j-1] + x[i+1,j+1]).
    sigma^4 is a Python double applied as a scalar multiply (HandCraftedModules.py:78).
    """
    xp = F.pad(x, (1, 1, 1, 1), "replicate")
    c = xp[:, :, 1:-1, 1:-1]
    gxx = xp[:, :, 1:-1, :-2] - 2.0 * c + xp[:, :, 1:-1, 2:]
    gyy = xp[:, :, :-2, 1:-1] - 2.0 * c + xp[:, :, 2:, 1:-1]
    gx = 0.5 * xp[:, :, :, :-2] - 0.5 * xp[:, :, :, 2:]          # [.., h+2, w]
    gxy = 0.5 * gx[:, :, :-2, :] - 0.5 * gx[:, :, 2:, :]
    return torch.abs(gxx * gyy - gxy * gxy) * (sigma ** 4)


# ----------------------------------------------------------------------------------------------
# a4/a5  3x3x3 NMS + soft-argmax + LAF composition           HandCraftedModules.py:208-291
# ----------------------------------------------------------------------------------------------

NMS_EPS = 1e-5  # HandCraftedModules.py:212


def float_to_u8_cpu(v):
    """float32 -> uint8 the way torch-CPU `.byte()` does it (truncate, wrap mod 256; Q4)."""
    return (np.trunc(v.astype(np.float64)).astype(np.int64) & 0xFF).astype(np.uint8)


def nms3d_mask(low, cur, high):
    """NMS3d on the middle slice (HandCraftedModules.py:208-220, :248): fp32 (x - m + eps) > 0,
    m = max over the 3x3x3 neighbourhood, spatial padding -inf, depth unpadded."""
    stack = torch.cat([low, cur, high], dim=1)                  # [1,3,h,w]
    m = F.max_pool2d(stack, 3, stride=1, padding=1).max(dim=1, keepdim=True)[0]
    return ((cur - m + NMS_EPS) > 0).float() * cur


def soft_argmax_weights(scales):
    """The [3,3,3,3] weight of HandCraftedModules.py:266-271 built from Utils.py:116-138:
    out channel c in (sigma, y, x); in channel d in (low,cur,high); offsets [-0.5,0.5,1.5] (Q2)."""
    off = torch.linspace(-3 / 2 + 1, 3 / 2, 3)                  # Utils.py:118 with w=3
    g = torch.zeros(3, 3, 3, 3)
    for d in range(3):
        g[0, d, :, :] = float(np.float32(scales[d]))            # torch.FloatTensor(scales)
        for i in range(3):
            g[1, d, i, :] = off[i]
            g[2, d, :, i] = off[i]
    return g


def nms3d_and_compose(low, cur, high, num_features, octave_map, scales, mrSize):
    """NMS3dAndComposeA.forward (HandCraftedModules.py:240-291).

    low/cur/high: float32 [1,1,h,w]; octave_map: uint8 numpy [h,w].  Returns
    (resp[n], LAFs[n,2,3] normalised, new_octave_map, flat_idxs[n]) or (None, None, octave_map, None).
    """
    h, w = cur.size(2), cur.size(3)
    nmsed = nms3d_mask(low, cur, high).clone()
    b = int(mrSize)
    if b < w and b < h:                                          # Utils.py:140-148
        nmsed[:, :, :b, :] = 0; nmsed[:, :, h - b:, :] = 0
        nmsed[:, :, :, :b] = 0; nmsed[:, :, :, w - b:] = 0
    else:
        nmsed = nmsed * 0
    om = torch.from_numpy(octave_map.astype(np.float32)).view(1, 1, h, w)
    nmsed = nmsed * (1.0 - om)
    n_pos = int((nmsed > 0).sum().item())
    if n_pos <= 1:
        return None, None, octave_map, None
    new_map = float_to_u8_cpu((om + nmsed).numpy().reshape(h, w))
    flat = nmsed.view(-1)
    if 0 < num_features < n_pos:
        vals, idxs = torch.topk(flat, k=num_features)
    else:
        idxs = flat.nonzero().view(-1)
        vals = flat[idxs]
    resp3d = torch.cat([low, cur, high], dim=1)
    num = F.conv2d(resp3d, soft_argmax_weights(scales), padding=1)
    den = F.conv2d(resp3d, torch.ones(3, 3, 3, 3), padding=1) + 1e-8
    sc_y_x = num / den
    ys = torch.arange(h, dtype=torch.float32).view(h, 1).expand(h, w)
    xs = torch.arange(w, dtype=torch.float32).view(1, w).expand(h, w)
    sc_y_x[0, 1] += ys
    sc_y_x[0, 2] += xs
    s = sc_y_x.view(3, -1).t()[idxs, :].clone()
    min_size = float(min(h, w))
    s[:, 0] = s[:, 0] / min_size
    s[:, 1] = s[:, 1] / float(h)
    s[:, 2] = s[:, 2] / float(w)
    LAFs = torch.zeros(s.size(0), 2, 3)
    LAFs[:, 0, 0] = s[:, 0]; LAFs[:, 1, 1] = s[:, 0]            # LAF.py:431-441
    LAFs[:, 0, 2] = s[:, 2]; LAFs[:, 1, 2] = s[:, 1]
    return vals, LAFs, new_map, idxs


# ----------------------------------------------------------------------------------------------
# a6  Multi-scale detector                                   SparseImgRepresenter.py:53-111
# ----------------------------------------------------------------------------------------------


def multi_scale_detector(pyr, sigmas, num_features, mrSize, th=0.0, return_levels=False):
    """Returns (resp[M], LAFs[M,2,3] normalised, pyr_idxs[M], level_idxs[M]) (+ per-level dump)."""
    resps, lafs, pidx, lidx, dump = [], [], [], [], []
    for o in range(len(pyr)):
        octave = pyr[o]
        h, w = octave[0].size(2), octave[0].size(3)
        omap = np.zeros((h, w), np.uint8)
        maps = [torch.clamp(hessian_response(octave[l], sigmas[o][l]) - th, min=0) for l in range(len(octave))]
        for l in range(1, len(octave) - 1):
            r, A, omap, idxs = nms3d_and_compose(maps[l - 1], maps[l], maps[l + 1], num_features, omap,
                                                 sigmas[o][l - 1:l + 2], mrSize)
            dump.append((o, l, None if r is None else idxs.clone(), None if r is None else r.clone()))
            if r is None:
                continue
            resps.append(r); lafs.append(A)
            pidx.append(torch.full((r.numel(),), float(o)))
            lidx.append(torch.full((r.numel(),), float(l - 1)))  # patches come from the level below
    resp = torch.cat(resps); LAFs = torch.cat(lafs); pidx = torch.cat(pidx); lidx = torch.cat(lidx)
    if 0 < num_features < resp.numel():
        resp, idxs = torch.topk(resp, k=num_features)
        LAFs, pidx, lidx = LAFs[idxs], pidx[idxs], lidx[idxs]
    if return_levels:
        return resp, LAFs, pidx, lidx, dump
    return resp, LAFs, pidx, lidx


# ----------------------------------------------------------------------------------------------
# a7/a8  Affine bilinear sampler                              LAF.py:313-390
# ----------------------------------------------------------------------------------------------


def extract_patches(img, LAFs, PS=32):
    """Closed form of affine_grid + grid_sample (bilinear, zeros, align_corners=False).

    out[n,0,i,j] = bilinear(img, p - 0.5), p = A_px (x_j, y_i)^T + t_px, x_j = (2j+1)/PS - 1,
    A_px = LAF[:, :, :2]*min(h,w), t_px = (LAF_x*w, LAF_y*h)   (LAF.py:313-324, 364-372).
    img float32 [1,1,h,w]; LAFs float32 [n,2,3] normalised.  Evaluated in float64, returned fp32.
    """
    h, w = img.size(2), img.size(3)
    n = LAFs.size(0)
    L = LAFs.double()
    ms = float(min(h, w))
    base = (2.0 * torch.arange(PS, dtype=torch.float64) + 1.0) / PS - 1.0
    gx = base.view(1, 1, PS); gy = base.view(1, PS, 1)
    px = (L[:, 0, 0] * ms).view(n, 1, 1) * gx + (L[:, 0, 1] * ms).view(n, 1, 1) * gy + (L[:, 0, 2] * w).view(n, 1, 1) - 0.5
    py = (L[:, 1, 0] * ms).view(n, 1, 1) * gx + (L[:, 1, 1] * ms).view(n, 1, 1) * gy + (L[:, 1, 2] * h).view(n, 1, 1) - 0.5
    x0 = torch.floor(px); y0 = torch.floor(py)
    fx = px - x0; fy = py - y0
    im = img.view(h, w).double()

    def tap(yy, xx):
        ok = (yy >= 0) & (yy < h) & (xx >= 0) & (xx < w)
        v = im[yy.clamp(0, h - 1).long(), xx.clamp(0, w - 1).long()]
        return torch.where(ok, v, torch.zeros_like(v))

    out = (tap(y0, x0) * (1 - fx) * (1 - fy) + tap(y0, x0 + 1) * fx * (1 - fy)
           + tap(y0 + 1, x0) * (1 - fx) * fy + tap(y0 + 1, x0 + 1) * fx * fy)
    return out.float().view(n, 1, PS, PS)


def extract_patches_from_pyramid(pyr, pyr_idxs, level_idxs, LAFs, PS=32):
    """LAF.py:376-404: route each LAF to pyr[o][l] and sample there."""
    out = torch.zeros(LAFs.size(0), 1, PS, PS)
    for o in range(len(pyr)):
        for l in range(len(pyr[o])):
            sel = ((pyr_idxs == o) & (level_idxs == l)).nonzero().view(-1)
            if sel.numel():
                out[sel] = extract_patches(pyr[o][l], LAFs[sel], PS)
    return out


# ----------------------------------------------------------------------------------------------
# a9/a12/a16  The three small CNNs                 architectures.py:33-82,204-252; HardNet.py:61-101
# ----------------------------------------------------------------------------------------------

BN_EPS = 1e-5
AFFNET_CFG = [(1, 16, 1), (16, 16, 1), (16, 32, 2), (32, 32, 1), (32, 64, 2), (64, 64, 1)]
HARDNET_CFG = [(1, 32, 1), (32, 32, 1), (32, 64, 2), (64, 64, 1), (64, 128, 2), (128, 128, 1)]
CONV_IDX = [0, 3, 6, 9, 12, 15]


def input_norm(x):
    """(x - mean) / (std_unbiased + 1e-7) per patch (architectures.py:231-235, HardNet.py:92-96)."""
    flat = x.view(x.size(0), -1)
    mp = flat.mean(dim=1).view(-1, 1, 1, 1)
    sp = flat.std(dim=1).view(-1, 1, 1, 1) + 1e-7
    return (x - mp) / sp


def _trunk(x, sd, cfg):
    for i, (cin, cout, stride) in zip(CONV_IDX, cfg):
        x = F.conv2d(x, sd["features.%d.weight" % i], stride=stride, padding=1)
        m = sd["features.%d.running_mean" % (i + 1)].view(1, -1, 1, 1)
        v = sd["features.%d.running_var" % (i + 1)].view(1, -1, 1, 1)
        x = F.relu((x - m) / torch.sqrt(v + BN_EPS))
    return x


def rectify_up_is_up(A):
    """LAF.py:285-291."""
    det = torch.sqrt(torch.abs(A[:, 0, 0] * A[:, 1, 1] - A[:, 1, 0] * A[:, 0, 1] + 1e-10))
    b2a2 = torch.sqrt(A[:, 0, 1] * A[:, 0, 1] + A[:, 0, 0] * A[:, 0, 0])
    out = torch.zeros_like(A)
    out[:, 0, 0] = b2a2 / det
    out[:, 1, 0] = (A[:, 1, 1] * A[:, 0, 1] + A[:, 1, 0] * A[:, 0, 0]) / (b2a2 * det)
    out[:, 1, 1] = det / b2a2
    return out


def affnet_raw(patches, sd):
    """tanh(conv8x8(trunk)) -> [n,3] (architectures.py:207-230)."""
    x = _trunk(input_norm(patches), sd, AFFNET_CFG)
    x = F.conv2d(x, sd["features.19.weight"], sd["features.19.bias"])
    return torch.tanh(x).view(-1, 3)


def affnet_forward(patches, sd):
    """AffNetFast.forward (architectures.py:247-252): [n,1,32,32] -> [n,2,2]."""
    xy = affnet_raw(patches, sd)
    A = torch.zeros(xy.size(0), 2, 2)
    A[:, 0, 0] = 1.0 + xy[:, 0]; A[:, 1, 0] = xy[:, 1]; A[:, 1, 1] = 1.0 + xy[:, 2]
    return rectify_up_is_up(A)


def orinet_raw(patches, sd):
    """OriNetFast trunk + 8x8 head with padding=1 -> 3x3 map -> tanh -> mean (architectures.py:36-59)."""
    x = _trunk(input_norm(patches), sd, AFFNET_CFG)
    x = F.conv2d(x, sd["features.19.weight"], sd["features.19.bias"], padding=1)
    return torch.tanh(x).mean(dim=(2, 3)).view(-1, 2)


def orinet_angle(patches, sd):
    xy = orinet_raw(patches, sd)
    return torch.atan2(xy[:, 0] + 1e-8, xy[:, 1] + 1e-8)       # architectures.py:78


def rotation_matrix(angle):
    """LAF.py:276-283: [[cos, sin], [-sin, cos]]."""
    c, s = torch.cos(angle), torch.sin(angle)
    R = torch.zeros(angle.numel(), 2, 2)
    R[:, 0, 0] = c; R[:, 0, 1] = s; R[:, 1, 0] = -s; R[:, 1, 1] = c
    return R


def orinet_forward(patches, sd):
    return rotation_matrix(orinet_angle(patches, sd))


def hardnet_forward(patches, sd):
    """HardNet.forward (HardNet.py:98-101): [n,1,32,32] -> L2-normalised [n,128]."""
    x = _trunk(input_norm(patches), sd, HARDNET_CFG)
    x = F.conv2d(x, sd["features.19.weight"])
    m = sd["features.20.running_mean"].view(1, -1, 1, 1)
    v = sd["features.20.running_var"].view(1, -1, 1, 1)
    x = ((x - m) / torch.sqrt(v + BN_EPS)).view(x.size(0), -1)
    return x / torch.sqrt((x * x).sum(dim=1, keepdim=True) + 1e-8)   # HardNet.py:12-19, eps 1e-8


# ----------------------------------------------------------------------------------------------
# a11  Affine-shape stage                                   SparseImgRepresenter.py:113-165
# ----------------------------------------------------------------------------------------------


def batch_eig2x2(A):
    """Utils.py:168-175."""
    trace = A[:, 0, 0] + A[:, 1, 1]
    delta1 = trace * trace - 4 * (A[:, 0, 0] * A[:, 1, 1] - A[:, 1, 0] * A[:, 0, 1])
    mask = (delta1 > 0).float()
    delta = torch.sqrt(torch.abs(delta1))
    l1 = mask * (trace + delta) / 2.0 + 1000.0 * (1.0 - mask)
    l2 = mask * (trace - delta) / 2.0 + 0.0001 * (1.0 - mask)
    return l1, l2


def check_touch_boundary(LAFs):
    """LAF.py:98-104: corners (+-1,+-1) through the normalised LAF must stay in [0,1] (Q5)."""
    pts = torch.tensor([[-1, -1, 1, 1], [-1, 1, -1, 1], [1, 1, 1, 1]], dtype=torch.float32)
    out = torch.matmul(LAFs, pts)                                # [n,2,4]
    bad = ((out > 1.0) | (out < 0.0)).sum(dim=(1, 2)) > 0
    return ~bad


def shape_filter_mask(base_A, new_LAFs):
    l1, l2 = batch_eig2x2(base_A)
    ratio = torch.abs(l1 / (l2 + 1e-8))
    return ((ratio < 6.0) & (ratio > (1.0 / 6.0))) & check_touch_boundary(new_LAFs)


def get_affine_shape(pyr, resp, LAFs, pyr_idxs, level_idxs, num_features, aff_sd, PS=32):
    """One AffNet iteration (num_Baum_iters=1), SparseImgRepresenter.py:113-165."""
    patches = extract_patches_from_pyramid(pyr, pyr_idxs, level_idxs, LAFs, PS)
    A = affnet_forward(patches, aff_sd)
    base_A = A                                                    # bmm(A, I)
    new_LAFs = torch.cat([torch.bmm(base_A, LAFs[:, :, 0:2]), LAFs[:, :, 2:]], dim=2)
    mask = shape_filter_mask(base_A, new_LAFs)
    n_ok = int(mask.sum().item())
    if num_features > 0 and n_ok > num_features:
        r, idxs = torch.topk(resp * mask.float(), k=num_features)
    else:
        idxs = mask.nonzero().view(-1)
        r = resp[idxs]
    out_LAFs = torch.cat([torch.bmm(base_A[idxs], LAFs[idxs][:, :, 0:2]), LAFs[idxs][:, :, 2:]], dim=2)
    return r, out_LAFs, pyr_idxs[idxs], level_idxs[idxs], dict(patches=patches, A=A, mask=mask, idxs=idxs)


def get_orientation(pyr, LAFs, pyr_idxs, level_idxs, ori_sd, PS=32):
    """SparseImgRepresenter.py:167-180 (the trailing re-extraction at :178 has no effect on the result).  ori_sd None = the
    constructor default OriNet=None: OrientationDetector(patch_size=19) on 19x19 patches, angle -> angles2A (LAF.py:180-186)."""
    if ori_sd is None:
        patches = extract_patches_from_pyramid(pyr, pyr_idxs, level_idxs, LAFs, 19)
        ang = orientation_hist(patches)
        c, s_ = torch.cos(ang).view(-1, 1, 1), torch.sin(ang).view(-1, 1, 1)
        R = torch.cat([torch.cat([c, s_], dim=2), torch.cat([-s_, c], dim=2)], dim=1)
    else:
        patches = extract_patches_from_pyramid(pyr, pyr_idxs, level_idxs, LAFs, PS)
        R = orinet_forward(patches, ori_sd)
    return torch.cat([torch.bmm(LAFs[:, :, :2], R), LAFs[:, :, 2:]], dim=2), dict(patches=patches, R=R)


# ----------------------------------------------------------------------------------------------
# a14/a15  LAF (de)normalisation and descriptor-level selection      LAF.py:407-429, 450-472
# ----------------------------------------------------------------------------------------------


def denormalize_lafs(LAFs, w, h):
    coef = torch.full((1, 2, 3), float(min(h, w)))
    coef[0, 0, 2] = float(w); coef[0, 1, 2] = float(h)
    return coef * LAFs


def normalize_lafs(LAFs, w, h):
    coef = torch.full((1, 2, 3), 1.0) / float(min(h, w))
    coef[0, 0, 2] = 1.0 / float(w); coef[0, 1, 2] = 1.0 / float(h)
    return coef * LAFs


def level_candidates(sigmas, pix_dists):
    """Octave-major list of sigma_l * 2^o in float64 (LAF.py:458-461)."""
    cand, octs, lvls = [], [], []
    for o in range(len(sigmas)):
        cand += list(np.array(sigmas[o]) * np.array(pix_dists[o]))
        octs += [o] * len(sigmas[o])
        lvls += list(range(len(sigmas[o])))
    return np.array(cand, dtype=np.float64), np.array(octs), np.array(lvls)


def pyramid_level_for_lafs(dLAFs, sigmas, pix_dists, PS):
    """LAF.py:450-472: scale = sqrt(|det A| + 1e-12) (fp32), needed = scale/PS (fp32), argmin of
    |cand - needed| in float64, first minimum wins."""
    scale = torch.sqrt(torch.abs(dLAFs[:, 0, 0] * dLAFs[:, 1, 1] - dLAFs[:, 0, 1] * dLAFs[:, 1, 0]) + 1e-12)
    needed = (scale / PS).numpy().astype(np.float64)
    cand, octs, lvls = level_candidates(sigmas, pix_dists)
    closest = np.abs(cand.reshape(-1, 1) - needed.reshape(1, -1)).argmin(axis=0)
    return torch.from_numpy(octs[closest]).float(), torch.from_numpy(lvls[closest]).float()


# ----------------------------------------------------------------------------------------------
# End-to-end (forward + extract_patches_from_pyr + HardNet)   SparseImgRepresenter.py:181-209
# ----------------------------------------------------------------------------------------------


def detect(x, aff_sd, ori_sd=None, num_features=2000, border=5, mrSize=5.192, nlevels=3, init_sigma=1.6,
           do_ori=False, debug=False):
    """ScaleSpaceAffinePatchExtractor.forward with num_Baum_iters=1, th=None.
    Returns (dLAFs[N,2,3] px units, responses[N], state) ; state carries pyr/sigmas/pix_dists."""
    pyr, sigmas, pix = scale_pyramid(x, nlevels, init_sigma, border)
    pre = int(1.5 * num_features)
    resp, LAFs, pidx, lidx = multi_scale_detector(pyr, sigmas, pre, mrSize)
    LAFs = LAFs.clone()
    LAFs[:, 0:2, 0:2] = mrSize * LAFs[:, :, 0:2]
    dbg = dict(det_resp=resp.clone(), det_LAFs=LAFs.clone(), det_pidx=pidx.clone(), det_lidx=lidx.clone())
    resp, LAFs, pidx, lidx, d1 = get_affine_shape(pyr, resp, LAFs, pidx, lidx, num_features, aff_sd)
    dbg.update(aff=d1, aff_LAFs=LAFs.clone())
    if do_ori:
        LAFs, d2 = get_orientation(pyr, LAFs, pidx, lidx, ori_sd)
        dbg.update(ori=d2)
    dLAFs = denormalize_lafs(LAFs, x.size(3), x.size(2))
    state = dict(pyr=pyr, sigmas=sigmas, pix_dists=pix, pyr_idxs=pidx, level_idxs=lidx)
    if debug:
        state["debug"] = dbg
    return dLAFs, resp, state


def describe(dLAFs, state, hard_sd, PS=32):
    """extract_patches_from_pyr (SparseImgRepresenter.py:181-188) + HardNet."""
    pyr = state["pyr"]
    o, l = pyramid_level_for_lafs(dLAFs, state["sigmas"], state["pix_dists"], PS)
    nl = normalize_lafs(dLAFs, pyr[0][0].size(3), pyr[0][0].size(2))
    patches = extract_patches_from_pyramid(pyr, o, l, nl, PS)
    return hardnet_forward(patches, hard_sd), patches, (o, l)


def detect_and_describe(x, aff_sd, ori_sd, hard_sd, num_features=2000, border=5, mrSize=5.192, do_ori=True):
    dLAFs, resp, state = detect(x, aff_sd, ori_sd, num_features, border, mrSize, do_ori=do_ori)
    desc, patches, _ = describe(dLAFs, state, hard_sd)
    return dLAFs, resp, desc


# ----------------------------------------------------------------------------------------------
# Synthetic inputs and weights shared by tests / bench (no reference counterpart)
# ----------------------------------------------------------------------------------------------


def synthetic_image(H, W, seed):
    """SURVEY.md §8(d) config 3: U[0,255) noise blurred with sigma=2, stretched to 0..255."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(1, 1, H, W, generator=g) * 255.0
    k1 = torch.from_numpy(gauss_kernel_1d(2.0).astype(np.float32))
    k = k1.numel()
    x = F.conv2d(F.pad(x, (k // 2, k // 2, 0, 0), "replicate"), k1.view(1, 1, 1, k))
    x = F.conv2d(F.pad(x, (0, 0, k // 2, k // 2), "replicate"), k1.view(1, 1, k, 1))
    x = (x - x.min()) / (x.max() - x.min()) * 255.0
    return x.contiguous()


def random_state_dict(kind, seed):
    """Random-init weights with the checkpoint layout (kind in affnet|orinet|hardnet).  Orthogonal-ish
    scale so activations stay O(1); running stats random but positive variance."""
    g = torch.Generator().manual_seed(seed)
    cfg = HARDNET_CFG if kind == "hardnet" else AFFNET_CFG
    sd = {}
    for i, (cin, cout, _s) in zip(CONV_IDX, cfg):
        sd["features.%d.weight" % i] = torch.randn(cout, cin, 3, 3, generator=g) * (0.9 / math.sqrt(9 * cin)) * 1.4
        sd["features.%d.running_mean" % (i + 1)] = torch.randn(cout, generator=g) * 0.1
        sd["features.%d.running_var" % (i + 1)] = torch.rand(cout, generator=g) * 0.5 + 0.5
    c = cfg[-1][1]
    if kind == "hardnet":
        sd["features.19.weight"] = torch.randn(128, c, 8, 8, generator=g) * (1.0 / math.sqrt(64 * c))
        sd["features.20.running_mean"] = torch.randn(128, generator=g) * 0.1
        sd["features.20.running_var"] = torch.rand(128, generator=g) * 0.5 + 0.5
    else:
        nout = 3 if kind == "affnet" else 2
        sd["features.19.weight"] = torch.randn(nout, c, 8, 8, generator=g) * (0.5 / math.sqrt(64 * c))
        sd["features.19.bias"] = torch.full((nout,), 0.01)
    return sd


# ----------------------------------------------------------------------------------------------
# §8(f) "next" rows: hand-crafted orientation and Baumberg affine shape   HandCraftedModules.py:81-192
# ----------------------------------------------------------------------------------------------


def circular_gauss_kernel(kernlen, sigma=None):
    """CircularGaussKernel(kernlen=..., sigma=...) with circ_zeros=False, norm=True (Utils.py:92-114), float64."""
    half = kernlen / 2
    r2 = float(half * half)
    sigma2 = 0.9 * r2 if sigma is None else 2.0 * sigma * sigma
    x = np.linspace(-half, half, kernlen)
    xv, yv = np.meshgrid(x, x, sparse=False, indexing="xy")
    k = np.exp(-((xv ** 2 + yv ** 2) / sigma2))
    return k / np.sum(k)


def orientation_hist_bins(patches, num_bins=36):
    """The smoothed 36-bin histogram of OrientationDetector.forward (HandCraftedModules.py:168-190) -> [n,36].
    gx/gy = (0.5,0,-0.5) cross-correlations with replicate padding; only the lower-bin weight wo0 is accumulated (as the
    reference does); smoothing (0.33,0.34,0.33) with ZERO padding."""
    PS = patches.size(2)
    x = patches
    xp = F.pad(x, (1, 1, 0, 0), "replicate")
    gx = 0.5 * xp[:, :, :, :-2] - 0.5 * xp[:, :, :, 2:]
    yp = F.pad(x, (0, 0, 1, 1), "replicate")
    gy = 0.5 * yp[:, :, :-2, :] - 0.5 * yp[:, :, 2:, :]
    gk = 10.0 * torch.from_numpy(circular_gauss_kernel(PS).astype(np.float32))
    mag = torch.sqrt(gx * gx + gy * gy + 1e-10) * gk
    ori = torch.atan2(gy, gx)
    o_big = float(num_bins) * (ori + 1.0 * math.pi) / (2.0 * math.pi)
    bo0 = torch.floor(o_big)
    wo1 = o_big - bo0
    bo0 = bo0 % num_bins
    wo0 = (1.0 - wo1) * mag
    bins = torch.stack([((bo0 == i).float() * wo0).mean(dim=(1, 2, 3)) for i in range(num_bins)], dim=1)   # [n,36]
    return F.conv1d(bins.view(-1, 1, num_bins), torch.tensor([[[0.33, 0.34, 0.33]]]), padding=1).view(-1, num_bins)


def orientation_hist(patches, num_bins=36):
    """OrientationDetector.forward (HandCraftedModules.py:168-192), returns the angle [n]: argmax of the smoothed histogram;
    angle = -(2 pi idx/36 - pi)."""
    idx = orientation_hist_bins(patches, num_bins).max(1)[1]
    return -((2.0 * float(np.pi) * idx.float() / float(num_bins)) - float(math.pi))


def baumberg_shape(patches):
    """AffineShapeEstimator.forward (HandCraftedModules.py:94-132): second-moment matrix -> inverse square root -> up-is-up."""
    PS = patches.size(2)
    x = patches
    xp = F.pad(x, (1, 1, 0, 0), "replicate")
    gx = xp[:, :, :, 2:] - xp[:, :, :, :-2]
    yp = F.pad(x, (0, 0, 1, 1), "replicate")
    gy = yp[:, :, 2:, :] - yp[:, :, :-2, :]
    gk = torch.from_numpy(circular_gauss_kernel(PS, sigma=(PS / 2) / 3.0).astype(np.float32))
    a = (gx * gx * gk).view(x.size(0), -1).mean(dim=1)
    b = (gx * gy * gk).view(x.size(0), -1).mean(dim=1)
    c = (gy * gy * gk).view(x.size(0), -1).mean(dim=1)
    eps = 1e-12
    mask = (b != 0).float()
    r1 = mask * (c - a) / (2.0 * b + eps)
    t1 = torch.sign(r1) / (torch.abs(r1) + torch.sqrt(1.0 + r1 * r1))
    r = 1.0 / torch.sqrt(1.0 + t1 * t1)
    t = t1 * r
    r = r * mask + 1.0 * (1.0 - mask)
    t = t * mask
    xx = 1.0 / torch.sqrt(r * r * a - 2.0 * r * t * b + t * t * c)
    zz = 1.0 / torch.sqrt(t * t * a + 2.0 * r * t * b + r * r * c)
    d = torch.sqrt(xx * zz)
    xx = xx / d
    zz = zz / d
    na = r * r * xx + t * t * zz
    nb = -r * t * xx + t * r * zz
    nc = t * t * xx + r * r * zz
    A = torch.zeros(x.size(0), 2, 2)
    A[:, 0, 0] = na; A[:, 0, 1] = nb; A[:, 1, 0] = nb; A[:, 1, 1] = nc
    return rectify_up_is_up(A)


def distance_matrix_vector(anchor, positive):
    """Losses.py:5-13."""
    d1 = torch.sum(anchor * anchor, dim=1).unsqueeze(-1)
    d2 = torch.sum(positive * positive, dim=1).unsqueeze(-1)
    return torch.sqrt((d1.repeat(1, positive.size(0)) + torch.t(d2.repeat(1, anchor.size(0))) - 2.0 * torch.mm(anchor, positive.t())) + 1e-6)


def match_snn(desc1, desc2, ratio=0.8):
    """train_AffNet_test_on_graffity.py:292-298: -> (idx_in_1, idx_in_2, min_dist, second_dist)."""
    dist = distance_matrix_vector(desc1, desc2)
    mn, idx2 = torch.min(dist, 1)
    dist[:, idx2] = 100000
    sec, _ = torch.min(dist, 1)
    mask = (mn / (sec + 1e-8)) <= ratio
    return torch.arange(idx2.size(0))[mask], idx2[mask], mn, sec


# ---------------------------------------------------------------------------------------------
# SURVEY 8(f) row 4: output formats
# ---------------------------------------------------------------------------------------------
def bsvd2x2(As):
    """Closed-form batched 2x2 SVD (LAF.py:106-144): U from atan2 on A A^T, V from atan2 on A^T A with the sign matrix of
    U^T A W folded in, singular values from the eigenvalues of A A^T.  Returns U, SIG, V as [n,2,2]."""
    As = As.float()
    Su = torch.bmm(As, As.permute(0, 2, 1))
    phi = 0.5 * torch.atan2(Su[:, 0, 1] + Su[:, 1, 0] + 1e-12, Su[:, 0, 0] - Su[:, 1, 1] + 1e-12)
    U = torch.zeros(As.size(0), 2, 2)
    U[:, 0, 0] = torch.cos(phi); U[:, 1, 1] = torch.cos(phi); U[:, 0, 1] = -torch.sin(phi); U[:, 1, 0] = torch.sin(phi)
    Sw = torch.bmm(As.permute(0, 2, 1), As)
    theta = 0.5 * torch.atan2(Sw[:, 0, 1] + Sw[:, 1, 0] + 1e-12, Sw[:, 0, 0] - Sw[:, 1, 1] + 1e-12)
    Wm = torch.zeros(As.size(0), 2, 2)
    Wm[:, 0, 0] = torch.cos(theta); Wm[:, 1, 1] = torch.cos(theta); Wm[:, 0, 1] = -torch.sin(theta); Wm[:, 1, 0] = torch.sin(theta)
    SUsum = Su[:, 0, 0] + Su[:, 1, 1]
    SUdif = torch.sqrt((Su[:, 0, 0] - Su[:, 1, 1]) ** 2 + 4 * Su[:, 0, 1] * Su[:, 1, 0] + 1e-12)
    SIG = torch.zeros(As.size(0), 2, 2)
    SIG[:, 0, 0] = torch.sqrt((SUsum + SUdif) / 2.0)
    SIG[:, 1, 1] = torch.sqrt((SUsum - SUdif) / 2.0)
    S = torch.bmm(torch.bmm(U.permute(0, 2, 1), As), Wm)
    C = torch.sign(S)
    C[:, 0, 1] = 0; C[:, 1, 0] = 0
    return U, SIG, torch.bmm(Wm, C)


def lafs_to_ell_t(LAFs):
    """LAFs2ellT (LAF.py:35-51): [n,2,3] pixel LAFs -> [n,5] = (x, y, a, b, c) of the ellipse a u^2 + 2 b u v + c v^2 = 1,
    the Oxford-affine text format written by hesaffBaum.py:46-48."""
    LAFs = LAFs.float()
    n = LAFs.size(0)
    ell = torch.zeros(n, 5)
    if n == 0:
        return ell
    scale = torch.sqrt(LAFs[:, 0, 0] * LAFs[:, 1, 1] - LAFs[:, 0, 1] * LAFs[:, 1, 0] + 1e-10)
    u, Wd, _ = bsvd2x2(LAFs[:, 0:2, 0:2] / scale.view(-1, 1, 1))
    Wd = Wd.clone()
    Wd[:, 0, 0] = 1.0 / (scale * scale * Wd[:, 0, 0] ** 2)
    Wd[:, 1, 1] = 1.0 / (scale * scale * Wd[:, 1, 1] ** 2)
    A = torch.bmm(torch.bmm(u, Wd), u.permute(0, 2, 1))
    ell[:, 0] = LAFs[:, 0, 2]; ell[:, 1] = LAFs[:, 1, 2]
    ell[:, 2] = A[:, 0, 0]; ell[:, 3] = A[:, 0, 1]; ell[:, 4] = A[:, 1, 1]
    return ell


def _reproj_distance_matrix(anchor, positive):
    """distance_matrix_vector of ReprojectionStuff.py:78-86 (NOT the one of Losses.py): returns [len(positive), len(anchor)],
    sqrt(|d1 + d2 - 2 p a^T + 1e-12|) in fp32."""
    d1 = torch.sum(anchor * anchor, dim=1)
    d2 = torch.sum(positive * positive, dim=1)
    return torch.sqrt(torch.abs((d1.expand(positive.size(0), anchor.size(0)) + torch.t(d2.expand(anchor.size(0), positive.size(0)))
                                 - 2.0 * torch.mm(positive, torch.t(anchor))) + 1e-12))


def gt_correspondences(LAFs1, LAFs2, H1to2, dist_threshold=6.0):
    """get_GT_correspondence_indexes (ReprojectionStuff.py:126-137, centre part of reprojectLAFs :23-40): centres of LAFs2 are
    mapped through H1to2^-1 into image 1; because that module's distance matrix comes out transposed, row i is a centre of LAFs1
    and it counts as a true match when ANY reprojected centre of LAFs2 lies within dist_threshold px of it.
    Returns (min_dist[mask], index_in_1[mask], index_of_nearest_in_2[mask])."""
    Hinv = torch.inverse(H1to2.float())
    c2 = torch.cat([LAFs2[:, :, 2].float(), torch.ones(LAFs2.size(0), 1)], dim=1)          # [n,3]
    p = c2 @ Hinv.t()
    p = p[:, :2] / p[:, 2:3]
    dist = _reproj_distance_matrix(p, LAFs1[:, :, 2].float())
    mn, idx = torch.min(dist, 1)
    mask = mn <= dist_threshold
    return mn[mask], torch.arange(0, idx.size(0))[mask], idx[mask]


def match_and_verify(LAFs1, desc1, LAFs2, desc2, H1to2, ratio=0.8, px=6.0):
    """The reference's application test (train_AffNet_test_on_graffity.py:289-300): SNN matching, then the reprojection check on
    the tentative pairs.  Returns (n_tentatives, n_true)."""
    i1, i2, _, _ = match_snn(desc1, desc2, ratio)
    _, keep, _ = gt_correspondences(LAFs1[i1], LAFs2[i2], H1to2, px)
    return int(i1.numel()), int(keep.numel())
