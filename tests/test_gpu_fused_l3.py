"""GPU tests of AffNet / OriNet's conv layer 3 fused into the first tcgen05 kernel (tcx_first.cuh, L3 = 1): the fused kernel issues the
same MMAs in the same order as the unfused pair tcx_first_kernel + tcx_conv_kernel and applies the same epilogue arithmetic, so its
layer-3 activations, the nets' outputs and the batched pipeline's outputs must be bit-identical to the unfused path
(`ag_debug_fuse_l3` switches between the two)."""
import contextlib

import pytest
import torch

from helpers import gold, gray_from_rgb, load_weights

pytestmark = pytest.mark.gpu
DEV = "cuda"
W = load_weights()
L3_UNIT_BYTES = 32 * 256 * 2 * 2     # layer-3 output per patch: 32 channels x 16x16, fp16 hi + lo planes


@pytest.fixture(scope="module")
def L():
    import affnet_b200._lib as lib
    lib.lib()
    return lib


@pytest.fixture(scope="module")
def nets(L):
    from affnet_b200.architectures import AffNetFast, OriNetFast
    from affnet_b200.HardNet import HardNet
    a, o, h = AffNetFast(PS=32), OriNetFast(PS=32), HardNet()
    a.load_state_dict(W["affnet"]); o.load_state_dict(W["orinet"]); h.load_state_dict(W["hardnet"])
    a, o, h = a.eval().to(DEV), o.eval().to(DEV), h.eval().to(DEV)
    for m in (a, o, h):
        m.set_engine(L.ENGINE_TC2)
    return a, o, h


@contextlib.contextmanager
def fused(L, on):
    old = L.lib().ag_debug_fuse_l3(1 if on else 0)
    try:
        yield
    finally:
        L.lib().ag_debug_fuse_l3(old)


def patch_sets():
    g = torch.Generator().manual_seed(33)
    return [("graf", torch.from_numpy(gold("graf_crop.npz")["aff_patches"]).float())] + \
           [("rand%d" % n, torch.rand(n, 1, 32, 32, generator=g) * 255) for n in (1, 127, 513)]


def layer3(L, net, P, on):
    """Layer 3's output: the raw fp16 hi + lo planes (L_S1_16 layout, at the start of the workspace) and their fp32 decode."""
    lib = L.lib()
    n = P.size(0)
    ws_bytes = lib.ag_net_workspace_bytes(net.KIND, n)
    ws = torch.full((ws_bytes,), 0xA5, dtype=torch.uint8, device=DEV)
    out = torch.full((n, 32, 16, 16), float("nan"), device=DEV)
    Pd = P.to(DEV).contiguous()
    with fused(L, on):
        L.check(lib.ag_debug_tcx_layer(net.handle(), L.ptr(Pd), n, 3, L.ptr(out), L.ptr(ws), ws_bytes, L.stream_ptr()))
        torch.cuda.synchronize()
    return ws[:n * L3_UNIT_BYTES].cpu(), out.cpu()


@pytest.mark.parametrize("kind", ["affnet", "orinet"])
def test_fused_layer3_bit_identical(L, nets, kind):
    net = dict(zip(("affnet", "orinet"), nets))[kind]
    for name, P in patch_sets():
        raw0, dec0 = layer3(L, net, P, False)
        raw1, dec1 = layer3(L, net, P, True)
        assert not torch.isnan(dec1).any(), (kind, name)
        assert torch.equal(raw0, raw1), (kind, name, int((raw0 != raw1).sum()))
        assert torch.equal(dec0, dec1), (kind, name)


def test_fused_nets_bit_identical(L, nets):
    aff, ori, _ = nets
    for name, P in patch_sets():
        Pd = P.to(DEV).contiguous()
        outs = []
        for on in (False, True):
            with fused(L, on):
                outs.append((aff(Pd), ori(Pd), ori(Pd, return_rot_matrix=False)))
                torch.cuda.synchronize()
        for a, b in zip(*outs):
            assert torch.equal(a, b), name


def test_fused_pipeline_bit_identical(L, nets):
    """The batched detect-and-describe pipeline (per-image keypoint counts, so some rows of the nets' batches are skipped)."""
    from affnet_b200.pipeline import DetectDescribePipeline
    aff, ori, hn = nets
    img = gray_from_rgb(gold("graf_crop.npz")["rgb"])
    imgs = torch.cat([img, img.flip(-1), img.flip(-2)]).to(DEV)
    res = []
    for on in (False, True):
        with fused(L, on):
            pipe = DetectDescribePipeline(imgs.size(0), imgs.size(2), imgs.size(3), aff, hn, ori, num_features=500, do_ori=True)
            res.append([t.clone() for t in pipe.run(imgs)])
            torch.cuda.synchronize()
    for a, b in zip(*res):
        assert torch.equal(a, b)
