"""Harness that imports the UNMODIFIED reference (ducha-aiki/affnet) from $AFFNET_REF, /root/reference or
baseline/_ref (first that holds SparseImgRepresenter.py) on CPU.  TEST INFRASTRUCTURE ONLY: used by
`tests/golden/make_golden.py` to generate the golden vectors that pin `oracle/affnet_oracle.py`, and by
bench.py's CPU leg when the reference tree is present.  Never imported by the product.

Shims (no edits to the reference): matplotlib stub (LAF.py:2 imports pyplot), map_location='cpu'
for checkpoints saved from CUDA, stdout silenced (the detector prints timings on every forward).
"""
import contextlib
import io
import os
import sys
import types

import numpy as np
import torch

def _find_ref():
    """Search order (SURVEY.md section 9): $AFFNET_REF, /root/reference, baseline/_ref next to the repository."""
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for c in (os.environ.get("AFFNET_REF"), "/root/reference", os.path.join(here, "baseline", "_ref")):
        if c and os.path.isfile(os.path.join(c, "SparseImgRepresenter.py")):
            return c
    return os.environ.get("AFFNET_REF", "/root/reference")


REF = _find_ref()


def available():
    return os.path.isfile(os.path.join(REF, "SparseImgRepresenter.py"))


_mods = None


def ref_modules():
    """Returns a dict of the reference's modules (imported once)."""
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise RuntimeError("reference tree not found at %s" % REF)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    for n in ("matplotlib", "matplotlib.pyplot"):
        if n not in sys.modules:
            sys.modules[n] = types.ModuleType(n)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    import importlib
    out = {}
    with contextlib.redirect_stdout(io.StringIO()):
        for n in ("Utils", "LAF", "HandCraftedModules", "SparseImgRepresenter", "architectures", "HardNet"):
            out[n] = importlib.import_module(n)
    _mods = out
    return out


def load_nets():
    m = ref_modules()
    aff = m["architectures"].AffNetFast(PS=32)
    aff.load_state_dict(torch.load(os.path.join(REF, "pretrained/AffNet.pth"), map_location="cpu")["state_dict"])
    ori = m["architectures"].OriNetFast(PS=32)
    ori.load_state_dict(torch.load(os.path.join(REF, "pretrained/OriNet.pth"), map_location="cpu")["state_dict"])
    hn = m["HardNet"].HardNet()
    hn.load_state_dict(torch.load(os.path.join(REF, "HardNet++.pth"), map_location="cpu")["state_dict"])
    return aff.eval(), ori.eval(), hn.eval()


def load_gray(path):
    """Same as train_AffNet_test_on_graffity.py:246-254 / hesaffnet.py:35-39."""
    from PIL import Image
    img = np.mean(np.array(Image.open(path).convert("RGB")), axis=2)
    t = torch.from_numpy(img.astype(np.float32))
    return t.view(1, 1, t.size(0), t.size(1))


def make_detector(aff, ori=None, num_features=2000, border=5, mrSize=5.192, th=None, nlevels=3):
    m = ref_modules()
    kw = dict(mrSize=mrSize, num_features=num_features, border=border, num_Baum_iters=1, AffNet=aff, nlevels=nlevels, th=th)
    if ori is not None:
        kw["OriNet"] = ori
    return m["SparseImgRepresenter"].ScaleSpaceAffinePatchExtractor(**kw)


def run_full(det, desc, img, do_ori):
    """train_AffNet_test_on_graffity.py:255-260 (get_geometry_and_descriptors)."""
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        LAFs, resp = det(img, do_ori=do_ori)
        patches = det.extract_patches_from_pyr(LAFs, PS=32)
        d = desc(patches)
    return LAFs, resp, patches, d
