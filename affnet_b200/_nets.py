"""Shared machinery of the three CNN modules: parameter containers with the checkpoint layout of the
reference, weight-blob packing and the ctypes forward calls."""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib as L

AFF_CFG = [(1, 16, 1), (16, 16, 1), (16, 32, 2), (32, 32, 1), (32, 64, 2), (64, 64, 1)]
HARD_CFG = [(1, 32, 1), (32, 32, 1), (32, 64, 2), (64, 64, 1), (64, 128, 2), (128, 128, 1)]


def make_features(cfg, head):
    """nn.Sequential with the reference's indices (features.0 conv, .1 bn, .2 relu, ... .18 dropout, .19 head ...)
    so that `load_state_dict(ckpt['state_dict'])` works unchanged."""
    layers = []
    for cin, cout, stride in cfg:
        layers += [nn.Conv2d(cin, cout, kernel_size=3, stride=stride, padding=1, bias=False),
                   nn.BatchNorm2d(cout, affine=False), nn.ReLU()]
    return nn.Sequential(*(layers + head))


class _NativeNet(nn.Module):
    KIND = None

    def __init__(self):
        super().__init__()
        self._handle = None
        self._handle_key = None
        self._engine = None   # None = library default (tensor cores for all three nets)

    # -- weights ------------------------------------------------------------------------------------------
    def _blob(self):
        sd = self.state_dict()
        parts = []
        for i in (0, 3, 6, 9, 12, 15):
            parts += [sd["features.%d.weight" % i], sd["features.%d.running_mean" % (i + 1)], sd["features.%d.running_var" % (i + 1)]]
        parts.append(sd["features.19.weight"])
        if self.KIND == L.NET_HARDNET:
            parts += [sd["features.20.running_mean"], sd["features.20.running_var"]]
        else:
            parts.append(sd["features.19.bias"])
        return torch.cat([p.detach().reshape(-1).float().cpu() for p in parts]).contiguous()

    def _version_key(self):
        return tuple((t.data_ptr(), t._version) for t in self.state_dict().values())

    def handle(self):
        """Opaque ag_net_t* with BatchNorm folded; rebuilt when parameters change."""
        key = self._version_key()
        if self._handle is None or key != self._handle_key:
            self._release()
            blob = self._blob()
            h = C.c_void_p()
            L.check(L.lib().ag_net_create(self.KIND, C.c_void_p(blob.data_ptr()), blob.numel(), C.byref(h)))
            self._handle, self._handle_key = h, key
            if self._engine is not None:
                L.check(L.lib().ag_net_set_engine(h, self._engine))
        return self._handle

    def set_engine(self, engine):
        """engine: L.ENGINE_TC2 (tcgen05 tensor-core engine, default), L.ENGINE_TC2_BF16 (HardNet with bf16 operands) or L.ENGINE_SIMT
        (exact fp32 CUDA cores); see include/affnet_b200.h.  Any other value raises AffnetB200Error once the net has a handle."""
        if self._handle is not None:
            L.check(L.lib().ag_net_set_engine(self._handle, engine))
        self._engine = engine
        return self

    @property
    def engine(self):
        return L.lib().ag_net_get_engine(self.handle())

    def _release(self):
        if self._handle is not None:
            try:
                L.lib().ag_net_destroy(self._handle)
            except Exception:
                pass
            object.__setattr__(self, "_handle", None)     # not nn.Module.__setattr__: at interpreter shutdown torch's globals may be gone

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _check_input(self, x):
        L.require_cuda(x, "input patches")
        if self.training:
            raise L.AffnetB200Error("affnet_b200 nets are inference-only: call .eval() first")
        if x.dim() != 4 or x.size(1) != 1 or x.size(2) != 32 or x.size(3) != 32:
            raise L.AffnetB200Error("expected patches of shape [n,1,32,32], got %s" % (tuple(x.shape),))
        return L.f32c(x)

    def _workspace(self, n, device):
        nbytes = L.lib().ag_net_workspace_bytes(self.KIND, n)
        return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes
