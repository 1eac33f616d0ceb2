"""GPU tests (-m gpu): the alternative kernel paths that a process selects once through the environment must give the SAME BITS as the
defaults, because they are what runs when a default cannot (no tensor-map encoder in the driver -> row-wise bulk copies in the blur;
a pyramid allocation beyond 2^31 elements -> the first register formulation of the detector).  Each variant runs in a subprocess (the
switches are read once per process) on the same seeded inputs and its pyramid / keypoints are compared with this process's."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")

_SCRIPT = r"""
import ctypes as C, sys, torch
sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[2] + "/tests")
import affnet_b200._lib as L
from affnet_b200.HandCraftedModules import ScalePyramid
g = torch.Generator().manual_seed(11)
x = torch.rand(2, 1, 480, 640, generator=g) * 255
k = torch.ones(1, 1, 5, 5) / 25
x = torch.nn.functional.conv2d(x, k, padding=2).cuda().contiguous()      # smooth enough to have stable extrema
sp = ScalePyramid(3, 1.6, 5)
plan, buf = sp.build(x)
lib = L.lib()
cap = 65536
ws_buf = torch.empty(lib.ag_detect_ws_bytes(C.byref(plan), cap), dtype=torch.uint8, device="cuda")
ws = L.DetectWs()
L.check(lib.ag_detect_ws_carve(C.byref(plan), cap, L.ptr(ws_buf), C.byref(ws)))
L.check(lib.ag_detect(C.byref(plan), L.ptr(buf), 0.0, 5, C.byref(ws), L.stream_ptr()))
nf = 1500
resp = torch.zeros(2, nf, device="cuda"); lafs = torch.zeros(2, nf, 2, 3, device="cuda")
oc = torch.zeros(2, nf, dtype=torch.int32, device="cuda"); lv = torch.zeros(2, nf, dtype=torch.int32, device="cuda")
cnt = torch.zeros(2, dtype=torch.int32, device="cuda")
L.check(lib.ag_select_keypoints(C.byref(plan), C.byref(ws), nf, 5.192, nf, L.ptr(resp), L.ptr(lafs), L.ptr(oc), L.ptr(lv), L.ptr(cnt), L.stream_ptr()))
torch.cuda.synchronize()
c = cnt.cpu()
for b in range(2):
    resp[b, int(c[b]):] = 0; lafs[b, int(c[b]):] = 0; oc[b, int(c[b]):] = 0; lv[b, int(c[b]):] = 0
torch.save({"pyr": buf.cpu(), "resp": resp.cpu(), "lafs": lafs.cpu(), "oc": oc.cpu(), "lv": lv.cpu(), "cnt": c}, sys.argv[1])
"""


def _run(tmp_path, name, env_extra):
    out = str(tmp_path / (name + ".pt"))
    env = dict(os.environ)
    for k in ("AG_BLUR_NO_TMA", "AG_DETECT_WARP_V1"):
        env.pop(k, None)
    env.update(env_extra)
    r = subprocess.run([sys.executable, "-c", _SCRIPT, out, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return torch.load(out)


def test_fallback_kernels_give_the_same_bits(tmp_path):
    base = _run(tmp_path, "default", {})
    assert int(base["cnt"].min()) > 200, base["cnt"]          # the input does produce keypoints
    for name, env in (("blur_rowwise_bulk", {"AG_BLUR_NO_TMA": "1"}), ("detector_v1", {"AG_DETECT_WARP_V1": "1"})):
        other = _run(tmp_path, name, env)
        for key in base:
            assert torch.equal(base[key], other[key]), (name, key)
