"""CPU tests (-m "not gpu") of the pipeline's estimator configuration: ag_pipeline_create_ex validates on the host and only borrows the
net handles (it never dereferences them), so its refusals, prefilter rule and workspace sizes are checked here without a device."""
import ctypes as C
import os

import pytest


@pytest.fixture(scope="module")
def L():
    import affnet_b200._lib as lib
    if not os.path.isfile(lib.LIB_PATH):
        lib.build()
    lib.lib()
    return lib


NET = C.c_void_p(0x1000)   # stands in for an ag_net_t*: create only stores it


def create(L, est, K=300, aff=NET, ori=NET, hard=NET, do_ori=1):
    cfg = L.PipelineConfig(2, 240, 320, K, 3, 5, 1.6, 5.192, do_ori, 0)
    h = C.c_void_p()
    rc = L.lib().ag_pipeline_create_ex(C.byref(cfg), C.byref(est) if est is not None else None, aff, ori, hard, C.byref(h))
    msg = L.lib().ag_last_error().decode()
    ws = L.lib().ag_pipeline_workspace_bytes(h) if rc == 0 else None
    if rc == 0:
        L.lib().ag_pipeline_destroy(h)
    return rc, msg, ws


def est(L, shape=0, n=1, sps=19, ori=1, ops=19):
    return L.PipelineEstimators(shape, n, sps, ori, ops)


def test_invalid_combinations_refused_with_message(L):
    cases = [
        (est(L, n=65), {}, "num_Baum_iters out of range"),
        (est(L, n=-1), {}, "num_Baum_iters out of range"),
        (est(L, shape=1, n=16, sps=42), {}, "Baumberg patch size out of range"),
        (est(L, shape=1, n=1, sps=2), {}, "Baumberg patch size out of range"),
        (est(L, ori=2, ops=42), {}, "orientation patch size out of range"),
        (est(L, ori=2, ops=2), {}, "orientation patch size out of range"),
        (est(L, shape=0, n=2), dict(aff=None), "needs an AffNet"),
        (est(L, ori=1), dict(ori=None), "AG_ORI_ORINET needs an OriNet"),
        (est(L, shape=2), {}, "unknown shape estimator"),
        (est(L, ori=3), {}, "unknown orientation estimator"),
    ]
    for e, kw, msg in cases:
        rc, text, _ = create(L, e, **kw)
        assert rc == -1 and msg in text, (e.shape, e.num_Baum_iters, e.shape_ps, e.ori, e.ori_ps, text)


def test_valid_combinations_and_defaults(L):
    # est == NULL is today's configuration; ag_pipeline_create is that call
    rc, _, ws_null = create(L, None)
    assert rc == 0
    rc, _, ws_default = create(L, est(L, shape=0, n=1, ori=1))
    assert rc == 0 and ws_default == ws_null
    cfg = L.PipelineConfig(2, 240, 320, 300, 3, 5, 1.6, 5.192, 1, 0)
    h = C.c_void_p()
    assert L.lib().ag_pipeline_create(C.byref(cfg), NET, NET, NET, C.byref(h)) == 0
    assert L.lib().ag_pipeline_workspace_bytes(h) == ws_null
    L.lib().ag_pipeline_destroy(h)
    # with est given, do_ori is ignored: OriNet mode needs the OriNet whatever do_ori says
    assert create(L, est(L, ori=1), ori=None, do_ori=0)[0] == -1
    assert create(L, est(L, ori=0), ori=None, do_ori=1)[0] == 0
    # no AffNet is needed without AffNet iterations; hand-crafted stages need no nets at all
    assert create(L, est(L, shape=0, n=0, ori=2), aff=None, ori=None)[0] == 0
    assert create(L, est(L, shape=1, n=16, sps=3, ori=2, ops=41), aff=None, ori=None)[0] == 0
    # AffNet x n > 1 carries the working LAFs and two more 2x2 buffers
    assert create(L, est(L, shape=0, n=2, ori=0))[2] > create(L, est(L, shape=0, n=1, ori=0))[2]
    assert create(L, est(L, shape=1, n=64, ori=0))[2] == create(L, est(L, shape=0, n=1, ori=0))[2]


def test_prefilter_limit_follows_num_baum_iters(L):
    """int(1.5 K) keypoints go through selection when there is a shape stage, K otherwise (SparseImgRepresenter.py:44)."""
    assert create(L, est(L, shape=1, n=1, ori=0), K=10923)[0] == 0
    assert create(L, est(L, shape=1, n=1, ori=0), K=10924)[0] == -3
    assert create(L, est(L, shape=1, n=0, ori=0), K=16384)[0] == 0
    assert create(L, est(L, shape=1, n=0, ori=0), K=16385)[0] == -3


def test_python_mode_selection():
    """DetectDescribePipeline picks the modes from the module types, as ScaleSpaceAffinePatchExtractor's constructor does."""
    import affnet_b200._lib as lib
    from affnet_b200.architectures import AffNetFast, OriNetFast
    from affnet_b200.HandCraftedModules import AffineShapeEstimator, OrientationDetector
    from affnet_b200.pipeline import _estimators
    e = _estimators(AffNetFast(PS=32), OriNetFast(PS=32), 1, True)
    assert (e.shape, e.num_Baum_iters, e.ori) == (lib.SHAPE_AFFNET, 1, lib.ORI_ORINET)
    e = _estimators(AffineShapeEstimator(patch_size=21), OrientationDetector(patch_size=17), 16, True)
    assert (e.shape, e.num_Baum_iters, e.shape_ps, e.ori, e.ori_ps) == (lib.SHAPE_BAUMBERG, 16, 21, lib.ORI_HIST, 17)
    e = _estimators(None, OrientationDetector(patch_size=19), 0, False)
    assert (e.num_Baum_iters, e.ori) == (0, lib.ORI_NONE)
    with pytest.raises(lib.AffnetB200Error):
        _estimators(OriNetFast(PS=32), None, 1, False)
    with pytest.raises(lib.AffnetB200Error):
        _estimators(AffNetFast(PS=32), AffNetFast(PS=32), 1, True)
