"""GPU tests of the tensor-core engine (ENGINE_TC2, tcx_first.cuh / tcx_conv.cuh): every conv layer's activations against the fp32
oracle (stage-isolated: `ag_debug_tcx_layer` decodes the engine's HBM layout), the three nets end to end, tile / pair / persistent-stride
invariance, and the engine selection."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import affnet_oracle as O
from helpers import gold, load_weights

pytestmark = pytest.mark.gpu
DEV = "cuda"
W = load_weights()


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


def oracle_layers(P, sd, cfg):
    """fp32 activations after conv layers 1..6 (BatchNorm + ReLU applied), as oracle/affnet_oracle.py::_trunk."""
    x = O.input_norm(P)
    out = []
    for i, (cin, cout, stride) in zip(O.CONV_IDX, cfg):
        x = F.conv2d(x, sd["features.%d.weight" % i], stride=stride, padding=1)
        m = sd["features.%d.running_mean" % (i + 1)].view(1, -1, 1, 1)
        v = sd["features.%d.running_var" % (i + 1)].view(1, -1, 1, 1)
        x = F.relu((x - m) / torch.sqrt(v + O.BN_EPS))
        out.append(x)
    return out


def patches():
    z = gold("graf_crop.npz")
    g = torch.Generator().manual_seed(8)
    return torch.cat([torch.from_numpy(z["aff_patches"])[:150], torch.rand(37, 1, 32, 32, generator=g) * 255])


@pytest.mark.parametrize("kind", ["affnet", "orinet", "hardnet"])
def test_tcx_layers_vs_oracle(L, nets, kind):
    """Layers 2..5 stage by stage (layer 1 is fused into the same kernel as layer 2).  AffNet / OriNet carry hi + lo planes: 2e-5 of
    the layer's largest activation; HardNet single fp16 planes: 2e-3 (one fp16 rounding of the stored value plus operand rounding).
    (A build with -DAG_AFF_LO8=1 stores AffNet's layer-2 residual plane as bytes: measured 1.9e-5 / 1.6e-5 / 2.8e-5 / 1.5e-5 on layers 2..5.)"""
    net = dict(zip(("affnet", "orinet", "hardnet"), nets))[kind]
    cfg = O.HARDNET_CFG if kind == "hardnet" else O.AFFNET_CFG
    P = patches()
    n = P.size(0)
    ref = oracle_layers(P, W[kind], cfg)
    lib = L.lib()
    ws_bytes = lib.ag_net_workspace_bytes(net.KIND, n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    Pd = P.to(DEV).contiguous()
    tol = 2e-3 if kind == "hardnet" else 2e-5
    for upto in (2, 3, 4, 5):
        r = ref[upto - 1]
        out = torch.full(r.shape, float("nan"), device=DEV)
        L.check(lib.ag_debug_tcx_layer(net.handle(), L.ptr(Pd), n, upto, L.ptr(out), L.ptr(ws), ws_bytes, L.stream_ptr()))
        torch.cuda.synchronize()
        d = (out.cpu() - r).abs()
        rel = d.max().item() / r.abs().max().item()
        print("\n%s layer %d %s: max|d| %.3e of max %.3e (rel %.2e), nan %d" % (kind, upto, tuple(r.shape), d.max().item(), r.abs().max().item(), rel, int(torch.isnan(out).sum())))
        assert not torch.isnan(out).any()
        assert rel < tol, (kind, upto, rel)


def test_tcx_nets_vs_oracle(L, nets):
    aff, ori, hn = nets
    z = gold("graf_crop.npz")
    g = torch.Generator().manual_seed(8)
    sets = [torch.from_numpy(z["aff_patches"]), torch.from_numpy(z["ori_desc_patches"]), torch.rand(37, 1, 32, 32, generator=g) * 255,
            torch.from_numpy(gold("face_patches.npz")["patches_u8"].astype(np.float32) / 255.0).view(-1, 1, 32, 32),
            torch.rand(300, 1, 32, 32, generator=g)]
    worst = [0.0, 0.0, 0.0, 0.0]
    for P in sets:
        Pd = P.to(DEV)
        dA = (aff(Pd).cpu() - O.affnet_forward(P, W["affnet"])).abs().max().item()
        dR = (ori(Pd).cpu() - O.orinet_forward(P, W["orinet"])).abs().max().item()
        dang = (ori(Pd, return_rot_matrix=False).cpu() - O.orinet_angle(P, W["orinet"]))
        dang = torch.atan2(torch.sin(dang), torch.cos(dang)).abs().max().item()
        dD = (hn(Pd).cpu() - O.hardnet_forward(P, W["hardnet"])).abs().max().item()
        worst = [max(a, b) for a, b in zip(worst, (dA, dR, dang, dD))]
    print("\nengine tc2: max|dA| %.2e  max|dR| %.2e  max|dangle| %.2e rad  max|ddesc| %.2e" % tuple(worst))
    assert worst[0] < 5e-5 and worst[1] < 1e-4 and worst[2] < 1e-4 and worst[3] < 6e-4, worst


def test_tcx_batching_invariance(L, nets):
    """Pairs of patches per tile in the 8x8 layers, 128 per head tile, persistent strides: a patch's result does not depend on its batch."""
    aff, ori, hn = nets
    g = torch.Generator().manual_seed(21)
    P = (torch.rand(513, 1, 32, 32, generator=g) * 255).to(DEV)
    for m in (aff, ori, hn):
        full = m(P)
        for lo, hi in ((0, 1), (1, 130), (130, 387), (386, 513), (512, 513), (3, 4)):
            assert torch.equal(m(P[lo:hi].contiguous()), full[lo:hi]), (type(m).__name__, lo, hi)


def test_raw_heads_vs_reference_torchscript(L):
    """f4 remainder: the raw head outputs (the contract of the reference's TorchScript exports) against goldens produced by running
    convertJIT/AffNetJIT.pt and OriNetJIT.pt on CPU (tests/golden/make_golden.py::make_jit)."""
    from affnet_b200.convertJIT import AffNetJIT, OriNetJIT
    z = gold("jit.npz")
    P = torch.from_numpy(z["patches"]).to(DEV)
    a, o = AffNetJIT(), OriNetJIT()
    a.load_state_dict(W["affnet"]); o.load_state_dict(W["orinet"])
    a, o = a.eval().to(DEV), o.eval().to(DEV)
    da = (a(P).cpu() - torch.from_numpy(z["affnet_raw"])).abs().max().item()
    do = (o(P).cpu() - torch.from_numpy(z["orinet_raw"])).abs().max().item()
    print("\nraw heads vs TorchScript goldens: AffNet %.2e, OriNet %.2e" % (da, do))
    assert a(P).shape == (P.size(0), 3) and o(P).shape == (P.size(0), 2)
    assert da < 2e-5 and do < 2e-5


def test_engine_selection(L, nets):
    """Engines 1, 2 and 3 (the first-generation tensor-core engine and its variants) do not exist: ag_net_set_engine refuses them and
    leaves the net's engine as it was.  0 (SIMT), 4 (tensor cores) and, for HardNet, 5 (bf16) select and run."""
    P = patches()[:40].to(DEV)
    for m in nets:
        ref = m(P)
        try:
            for e in (1, 2, 3):
                with pytest.raises(L.AffnetB200Error):
                    m.set_engine(e)
                assert m.engine == L.ENGINE_TC2
            engines = (L.ENGINE_SIMT, L.ENGINE_TC2, L.ENGINE_TC2_BF16) if m.KIND == L.NET_HARDNET else (L.ENGINE_SIMT, L.ENGINE_TC2)
            for e in engines:
                m.set_engine(e)
                assert m.engine == e
                assert (m(P) - ref).abs().max().item() < 1e-2, (type(m).__name__, e)
            if m.KIND != L.NET_HARDNET:
                with pytest.raises(L.AffnetB200Error):
                    m.set_engine(L.ENGINE_TC2_BF16)
        finally:
            m.set_engine(L.ENGINE_TC2)


def test_hardnet_bf16_engine(L):
    """BASELINE.json configs[4] asks for a bf16 HardNet tensor-core path: engine 5 = the second-generation engine with bf16 operands
    (activations bf16, weights bf16 + bf16 residual in layers 2-3, fp32 accumulate).  Own tolerance (SURVEY section 7 hard part 1: ~1e-2):
    bf16 keeps 8 mantissa bits, the emulation on the 2000 graf patches gives 1.6e-3 with exact weights and 7e-3 with plain bf16 weights."""
    from affnet_b200.HardNet import HardNet
    hn = HardNet(); hn.load_state_dict(W["hardnet"]); hn = hn.eval().to(DEV)
    hn.set_engine(L.ENGINE_TC2_BF16)
    z = gold("graf_crop.npz")
    g = torch.Generator().manual_seed(8)
    worst = 0.0
    for P in (torch.from_numpy(z["ori_desc_patches"]), torch.rand(300, 1, 32, 32, generator=g) * 255):
        d = hn(P.to(DEV)).cpu()
        assert ((d.norm(dim=1) - 1).abs() < 1e-4).all()
        worst = max(worst, (d - O.hardnet_forward(P, W["hardnet"])).abs().max().item())
    print("\nengine tc2-bf16 (HardNet): max|ddesc| %.2e" % worst)
    assert worst < 8e-3, worst
    hn.set_engine(L.ENGINE_TC2)
    assert (hn(P.to(DEV)).cpu() - O.hardnet_forward(P, W["hardnet"])).abs().max() < 6e-4      # and back
