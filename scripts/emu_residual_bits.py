"""Developer experiment (CPU, no GPU): how many bits do the residual ("lo") planes of AffNet / OriNet activations need?
fp64 forward of the two nets on the golden patches with the output of chosen layers quantised as fp16 only | fp16 + fp16 residual (what the
engine stores) | fp16 + fp8 residual (e5m2, or e4m3 scaled by 2^10).  Output: max / mean deviation of the head outputs from the unquantised
forward.  AffNet needs <= 5e-5 (OriNet amplifies its error 15x towards the 1e-3 LAF contract).    python scripts/emu_residual_bits.py

Second part: fewer MMAs per K step.  The engine computes every conv as A_hi W_hi + A_hi W_lo + A_lo W_hi (fp16 planes, weights scaled by a
power of two so that the largest is near 2^13).  Rows: that split itself; both correction products as one kind::f8f6f4 MMA with e5m2 A and B
(A_hi, A_lo, W_hi, W_lo rounded to e5m2 inside the correction) or e4m3 A (A_lo x 2^10) and e5m2 B, in layers 2-6 or layer 2 only; and the
weight residual dropped in one layer.  Deviations against the unquantised fp64 forward."""
import sys, torch, torch.nn.functional as F
import os
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import affnet_oracle as O
from helpers import gold, load_weights
W = load_weights()
torch.set_num_threads(8)
z = gold("graf_crop.npz")
g = torch.Generator().manual_seed(8)
P = torch.cat([torch.from_numpy(z["aff_patches"])[:300], torch.rand(50, 1, 32, 32, generator=g) * 255]).double()
for name, cfgname in (("affnet", "AFF"), ("orinet", "ORI")):
    sd = {k: v.double() for k, v in W[name].items()}
    cfg = [(1,16,1),(16,16,1),(16,32,2),(32,32,1),(32,64,2),(64,64,1)]
    def run(quant_after, q):
        x = O.input_norm(P.float()).double()
        for li, (i, (cin, cout, stride)) in enumerate(zip(O.CONV_IDX, cfg)):
            x = F.conv2d(x, sd["features.%d.weight" % i], stride=stride, padding=1)
            m = sd["features.%d.running_mean" % (i + 1)].view(1, -1, 1, 1); v = sd["features.%d.running_var" % (i + 1)].view(1, -1, 1, 1)
            x = F.relu((x - m) / torch.sqrt(v + O.BN_EPS))
            if li + 1 in quant_after: x = q(x)
        # head conv (8x8 -> 1x1) + tanh
        hi = [k for k in sd if k.endswith(".weight") and sd[k].dim() == 4][-1]
        y = F.conv2d(x, sd[hi], bias=sd.get(hi.replace("weight", "bias")))
        return torch.tanh(y).flatten(1)
    ident = lambda x: x
    def q_fp16(x): return x.half().double()
    def q_hi_lo16(x):
        h = x.half().double(); return h + (x - h).half().double()
    def q_hi_lo8(x):
        h = x.half().double(); return h + (x - h).float().to(torch.float8_e5m2).double()
    def q_hi_lo8m3(x):
        h = x.half().double(); r = (x - h).float() * 1024.0; return h + r.to(torch.float8_e4m3fn).double() / 1024.0
    ref = run((), ident)
    for label, layers, q in (("L2 out fp16 only", (2,), q_fp16), ("L2 out hi+lo16", (2,), q_hi_lo16), ("L2 out hi+lo e5m2", (2,), q_hi_lo8),
                             ("L2 out hi+lo e4m3*1024", (2,), q_hi_lo8m3),
                             ("all layers hi+lo16", (1,2,3,4,5), q_hi_lo16), ("L2,L4 hi+lo e5m2, rest lo16", None, None)):
        if layers is None:
            def run2():
                x = O.input_norm(P.float()).double()
                for li, (i, (cin, cout, stride)) in enumerate(zip(O.CONV_IDX, cfg)):
                    x = F.conv2d(x, sd["features.%d.weight" % i], stride=stride, padding=1)
                    m = sd["features.%d.running_mean" % (i + 1)].view(1, -1, 1, 1); v = sd["features.%d.running_var" % (i + 1)].view(1, -1, 1, 1)
                    x = F.relu((x - m) / torch.sqrt(v + O.BN_EPS))
                    if li + 1 in (2, 4): x = q_hi_lo8(x)
                    elif li + 1 in (1, 3, 5): x = q_hi_lo16(x)
                hi = [k for k in sd if k.endswith(".weight") and sd[k].dim() == 4][-1]
                return torch.tanh(F.conv2d(x, sd[hi], bias=sd.get(hi.replace("weight", "bias")))).flatten(1)
            out = run2()
        else:
            out = run(layers, q)
        print("%-8s %-28s max |d out| %.3e   mean %.3e" % (name, label, (out - ref).abs().max().item(), (out - ref).abs().mean().item()))


def h16(t): return t.half().double()
def q8(t, dt, s=1.0): return (t * s).float().to(dt).double() / s
E5, E4 = torch.float8_e5m2, torch.float8_e4m3fn
for name in ("affnet", "orinet"):
    sd = {k: v.double() for k, v in W[name].items()}
    cfg = [(1,16,1),(16,16,1),(16,32,2),(32,32,1),(32,64,2),(64,64,1)]
    def run_split(mode=None, layers=(), drop_w=()):
        """mode None: unquantised; "lo16": the engine's split; "e5e5" / "e4e5": fp8 correction products in `layers`; drop_w: no W_lo."""
        x = O.input_norm(P.float()).double()
        for li, (i, (cin, cout, stride)) in enumerate(zip(O.CONV_IDX, cfg)):
            w = sd["features.%d.weight" % i]
            c = lambda a, b: F.conv2d(a, b, stride=stride, padding=1)
            if mode is None:
                y = c(x, w)
            else:
                sc = 2.0 ** (13 - torch.floor(torch.log2(w.abs().max())).item())
                ws = w * sc
                ah, al, wh, wl = h16(x), x - h16(x), h16(ws), ws - h16(ws)
                if mode == "e5e5" and li + 1 in layers:
                    y = c(ah, wh) + c(q8(ah, E5), q8(wl, E5)) + c(q8(al, E5), q8(wh, E5))
                elif mode == "e4e5" and li + 1 in layers:
                    y = c(ah, wh) + c(q8(ah, E4), q8(wl, E5)) + c(q8(al, E4, 1024.0), q8(wh, E5, 1.0 / 1024))
                else:
                    y = c(ah, wh) + (0 if li + 1 in drop_w else c(ah, h16(wl))) + c(h16(al), wh)
                y = y / sc
            m = sd["features.%d.running_mean" % (i + 1)].view(1, -1, 1, 1); v = sd["features.%d.running_var" % (i + 1)].view(1, -1, 1, 1)
            x = F.relu((y - m) / torch.sqrt(v + O.BN_EPS))
        hk = [k for k in sd if k.endswith(".weight") and sd[k].dim() == 4][-1]
        return torch.tanh(F.conv2d(x, sd[hk], bias=sd.get(hk.replace("weight", "bias")))).flatten(1)
    ref = run_split()
    rows = [("split hi+lo16 (engine)", dict(mode="lo16")),
            ("fp8 corr e5m2/e5m2 L2-6", dict(mode="e5e5", layers=(2, 3, 4, 5, 6))),
            ("fp8 corr e4m3/e5m2 L2-6", dict(mode="e4e5", layers=(2, 3, 4, 5, 6))),
            ("fp8 corr e5m2/e5m2 L2", dict(mode="e5e5", layers=(2,))),
            ("fp8 corr e4m3/e5m2 L2", dict(mode="e4e5", layers=(2,)))] + \
           [("no W_lo in layer %d" % l, dict(mode="lo16", drop_w=(l,))) for l in (2, 3, 4, 5, 6)]
    for label, kw in rows:
        d = (run_split(**kw) - ref).abs()
        print("%-8s %-28s max |d out| %.3e   mean %.3e" % (name, label, d.max().item(), d.mean().item()))
