"""Batched detect-and-describe for B same-sized images (new API; the reference handles one image at a time):
the whole ScaleSpaceAffinePatchExtractor.forward + extract_patches_from_pyr + HardNet chain as one fixed kernel
sequence with device-side counters, optionally replayed as a CUDA graph."""
import ctypes as C

import torch

from . import _lib as L
from ._nets import _NativeNet
from .HandCraftedModules import AffineShapeEstimator, OrientationDetector


def _estimators(AffNet, OriNet, num_Baum_iters, do_ori):
    """The estimator modes of ScaleSpaceAffinePatchExtractor's constructor, chosen by module type: AffNet is an AffNetFast or an
    AffineShapeEstimator (may be None with num_Baum_iters=0); OriNet an OriNetFast or an OrientationDetector.  A missing net is left
    to the library, which refuses the combination with its message."""
    n = int(num_Baum_iters)
    if isinstance(AffNet, AffineShapeEstimator):
        shape, shape_ps = L.SHAPE_BAUMBERG, int(AffNet.PS)
    elif AffNet is None or (isinstance(AffNet, _NativeNet) and AffNet.KIND == L.NET_AFFNET):
        shape, shape_ps = L.SHAPE_AFFNET, 32
    else:
        raise L.AffnetB200Error("AffNet must be an AffNetFast, an AffineShapeEstimator or None, not %s" % type(AffNet).__name__)
    if not do_ori:
        ori, ori_ps = L.ORI_NONE, 0
    elif isinstance(OriNet, OrientationDetector):
        ori, ori_ps = L.ORI_HIST, int(OriNet.PS)
    elif OriNet is None or (isinstance(OriNet, _NativeNet) and OriNet.KIND == L.NET_ORINET):
        ori, ori_ps = L.ORI_ORINET, 32
    else:
        raise L.AffnetB200Error("OriNet must be an OriNetFast or an OrientationDetector, not %s" % type(OriNet).__name__)
    return L.PipelineEstimators(shape, n, shape_ps, ori, ori_ps)


def _handle(m):
    """ag_net_t of a CNN module; the hand-crafted estimators have none (the library derives their windows from the patch size)."""
    return m.handle() if isinstance(m, _NativeNet) else None


class DetectDescribePipeline:
    def __init__(self, B, H, W, AffNet, HardNet, OriNet=None, num_features=2000, border=5, mrSize=5.192, nlevels=3,
                 init_sigma=1.6, do_ori=True, cand_cap=0, device="cuda", outputs=None, num_Baum_iters=1):
        """outputs: optional list of (lafs [B,K,2,3], desc [B,K,128], count [B] int32) CUDA tensors, one tuple per output slot, that the
        kernels write into directly (e.g. DescriptorExchange.outputs(): the blocks an all-gather sends); default: one private slot.
        Estimators as ScaleSpaceAffinePatchExtractor selects them: AffNet = AffNetFast (num_Baum_iters AffNet iterations) or
        AffineShapeEstimator (num_Baum_iters Baumberg iterations), either or None with num_Baum_iters=0 (no shape stage); with do_ori,
        OriNet = OriNetFast or OrientationDetector (gradient histogram).  Patch sizes come from the modules."""
        self.cfg = L.PipelineConfig(B, H, W, num_features, nlevels, border, float(init_sigma), float(mrSize), 1 if do_ori else 0, cand_cap)
        self.est = _estimators(AffNet, OriNet, num_Baum_iters, do_ori)
        self.nets = (AffNet, OriNet, HardNet)  # keep the modules alive; the C pipeline only BORROWS their ag_net_t handles
        self._h = None
        self._net_handles = None
        self._bind_nets()
        self.B, self.H, self.W, self.K = B, H, W, num_features
        self.device = torch.device(device)
        self.ws_bytes = L.lib().ag_pipeline_workspace_bytes(self._h)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=self.device)
        if outputs is None:
            outputs = [(torch.empty(B, num_features, 2, 3, dtype=torch.float32, device=self.device),
                        torch.empty(B, num_features, 128, dtype=torch.float32, device=self.device),
                        torch.zeros(B, dtype=torch.int32, device=self.device))]
        for (l_, d_, c_) in outputs:
            if not (l_.is_contiguous() and d_.is_contiguous() and c_.is_contiguous() and l_.shape == (B, num_features, 2, 3)
                    and d_.shape == (B, num_features, 128) and c_.shape == (B,) and c_.dtype == torch.int32 and l_.dtype == torch.float32):
                raise L.AffnetB200Error("outputs: expected contiguous (lafs [B,K,2,3] f32, desc [B,K,128] f32, count [B] i32) per slot")
        self._slots = [(l_, torch.empty(B, num_features, dtype=torch.float32, device=self.device), d_, c_) for (l_, d_, c_) in outputs]
        self.lafs, self.resp, self.desc, self.count = self._slots[0]
        self._graphs = None
        self._graph = None
        self._static_in = None

    def _bind_nets(self):
        """(Re)create the C pipeline over the nets' CURRENT handles.  A module rebuilds (and frees) its ag_net_t when its parameters
        change (load_state_dict, .to(), in-place edits): the pipeline must never touch the freed handle, so every run()/replay() compares
        the handle objects it was built with against the modules' and rebinds (run) or refuses (replay: the captured graph holds the
        old weight pointers) when they differ."""
        AffNet, OriNet, HardNet = self.nets
        hs = (_handle(AffNet), _handle(OriNet), _handle(HardNet))
        if self._h is not None:
            L.lib().ag_pipeline_destroy(self._h)
            self._h = None
        h = C.c_void_p()
        L.check(L.lib().ag_pipeline_create_ex(C.byref(self.cfg), C.byref(self.est), hs[0], hs[1], hs[2], C.byref(h)))
        self._h, self._net_handles, self._graph = h, hs, None

    def _nets_current(self):
        return all(not isinstance(n, _NativeNet) or n._handle is h for n, h in zip(self.nets, self._net_handles))

    def __del__(self):
        try:
            L.lib().ag_pipeline_destroy(self._h)
        except Exception:
            pass

    @property
    def launches(self):
        return L.lib().ag_pipeline_launch_count(self._h)

    def run(self, imgs, slot=0):
        """imgs CUDA float32 [B,1,H,W] or [B,H,W] -> (lafs [B,K,2,3] px, resp [B,K], desc [B,K,128], count [B]) of output slot `slot`.
        Rows >= count[b] are unspecified.  No host synchronisation."""
        imgs = L.f32c(imgs, "imgs")
        if not self._nets_current() or any(isinstance(n, _NativeNet) and n.handle() is not h for n, h in zip(self.nets, self._net_handles)):
            self._bind_nets()      # a net was reloaded / moved since the pipeline was built
        if imgs.numel() != self.B * self.H * self.W:
            raise L.AffnetB200Error("expected %d x %d x %d pixels" % (self.B, self.H, self.W))
        lafs, resp, desc, count = self._slots[slot]
        L.check(L.lib().ag_pipeline_run(self._h, L.ptr(imgs), L.ptr(self.ws), self.ws_bytes, L.ptr(lafs), L.ptr(resp),
                                        L.ptr(desc), L.ptr(count), L.stream_ptr()))
        return lafs, resp, desc, count

    def check(self):
        """Synchronises and raises if any image overflowed the candidate capacity (count == -1)."""
        if any(bool((c < 0).any().item()) for (_, _, _, c) in self._slots):
            raise L.AffnetB200Error("candidate capacity exceeded: construct the pipeline with a larger cand_cap")
        return self

    def capture(self):
        """Capture one run() into a CUDA graph over a static input buffer; use replay(imgs) afterwards."""
        self._static_in = torch.zeros(self.B, 1, self.H, self.W, dtype=torch.float32, device=self.device)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.run(self._static_in)  # warm-up: sets kernel attributes outside capture
        torch.cuda.current_stream().wait_stream(s)
        self._graphs = []
        for slot in range(len(self._slots)):     # one graph per output slot (the output pointers are baked into the launches)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.run(self._static_in, slot)
            self._graphs.append(g)
        self._graph = self._graphs[0]
        return self

    def replay(self, imgs=None, slot=0):
        if self._graph is None:
            raise L.AffnetB200Error("call capture() first")
        if not self._nets_current():
            raise L.AffnetB200Error("a net of this pipeline was reloaded after capture(): the graph holds the old weights - call capture() again")
        if imgs is not None:
            self._static_in.copy_(imgs.view_as(self._static_in), non_blocking=True)
        self._graphs[slot].replay()
        return self._slots[slot]
