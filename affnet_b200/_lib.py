"""ctypes binding of the C ABI in include/affnet_b200.h (libaffnet_b200.so, sm_100a).

There is NO CPU / PyTorch fallback: if the shared library is missing or no sm_100 device is usable, every
entry point raises.  PyTorch is used only to own device memory and streams.
"""
import ctypes as C
import os
import subprocess

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AFFNET_B200_LIB", os.path.join(HERE, "lib", "libaffnet_b200.so"))   # override: developer builds only
AG_MAX_OCTAVES, AG_MAX_LEVELS = 16, 8
NET_AFFNET, NET_ORINET, NET_HARDNET = 0, 1, 2
ENGINE_SIMT, ENGINE_TC2, ENGINE_TC2_BF16 = 0, 4, 5


class AffnetB200Error(RuntimeError):
    pass


class PyramidPlan(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("H", C.c_int), ("W", C.c_int), ("n_octaves", C.c_int), ("n_levels", C.c_int),
        ("h", C.c_int * AG_MAX_OCTAVES), ("w", C.c_int * AG_MAX_OCTAVES),
        ("level_offset", (C.c_longlong * AG_MAX_LEVELS) * AG_MAX_OCTAVES),
        ("total_floats", C.c_longlong),
        ("sigma", (C.c_double * AG_MAX_LEVELS) * AG_MAX_OCTAVES),
        ("blur_sigma", (C.c_double * AG_MAX_LEVELS) * AG_MAX_OCTAVES),
        ("pix_dist", C.c_double * AG_MAX_OCTAVES),
    ]


class DetectWs(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("cand_cap", C.c_int), ("n_level_slots", C.c_int),
        ("d_cand_val", C.c_void_p), ("d_cand_seq", C.c_void_p), ("d_cand_scyx", C.c_void_p), ("d_cand_aux", C.c_void_p),
        ("d_cand_count", C.c_void_p), ("d_level_pos", C.c_void_p), ("d_level_emit", C.c_void_p), ("d_variants", C.c_void_p),
        ("d_octave_maps", C.c_void_p),
    ]


class PipelineConfig(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("H", C.c_int), ("W", C.c_int), ("num_features", C.c_int), ("nlevels", C.c_int),
        ("border", C.c_int), ("init_sigma", C.c_double), ("mrSize", C.c_double), ("do_ori", C.c_int),
        ("cand_cap", C.c_int),
    ]


SHAPE_AFFNET, SHAPE_BAUMBERG = 0, 1
ORI_NONE, ORI_ORINET, ORI_HIST = 0, 1, 2


class PipelineEstimators(C.Structure):
    _fields_ = [("shape", C.c_int), ("num_Baum_iters", C.c_int), ("shape_ps", C.c_int), ("ori", C.c_int), ("ori_ps", C.c_int)]


# name -> (restype, argtypes); every symbol declared in include/affnet_b200.h
vp, i32, f32, f64, sz = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_size_t
PROTOTYPES = {
    "ag_last_error": (C.c_char_p, []),
    "ag_abi_version": (i32, []),
    "ag_prof_begin": (i32, [vp]),
    "ag_prof_end": (i32, []),
    "ag_prof_get": (i32, [i32, C.POINTER(C.c_char_p), C.POINTER(f32)]),
    "ag_pyramid_plan": (i32, [i32, i32, i32, i32, f64, i32, C.POINTER(PyramidPlan)]),
    "ag_pyramid_build": (i32, [C.POINTER(PyramidPlan), vp, vp, vp]),
    "ag_gaussian_blur": (i32, [vp, vp, i32, i32, i32, f64, vp]),
    "ag_hessian_response": (i32, [vp, vp, i32, i32, i32, f64, f32, vp]),
    "ag_detect_ws_bytes": (sz, [C.POINTER(PyramidPlan), i32]),
    "ag_detect_ws_carve": (i32, [C.POINTER(PyramidPlan), i32, vp, C.POINTER(DetectWs)]),
    "ag_detect": (i32, [C.POINTER(PyramidPlan), vp, f32, i32, C.POINTER(DetectWs), vp]),
    "ag_detect_level_from_responses": (i32, [vp, vp, vp, i32, i32, C.POINTER(f64), i32, vp, vp, i32, C.POINTER(DetectWs), vp]),
    "ag_select_keypoints": (i32, [C.POINTER(PyramidPlan), C.POINTER(DetectWs), i32, f32, i32, vp, vp, vp, vp, vp, vp]),
    "ag_extract_patches": (i32, [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp]),
    "ag_extract_patches_pyr": (i32, [C.POINTER(PyramidPlan), vp, vp, vp, vp, vp, i32, i32, vp, vp]),
    "ag_pyramid_level_for_lafs": (i32, [C.POINTER(PyramidPlan), vp, i32, i32, vp, vp, vp]),
    "ag_net_create": (i32, [i32, vp, sz, C.POINTER(vp)]),
    "ag_net_destroy": (None, [vp]),
    "ag_net_blob_floats": (sz, [i32]),
    "ag_net_set_engine": (i32, [vp, i32]),
    "ag_net_get_engine": (i32, [vp]),
    "ag_net_workspace_bytes": (sz, [i32, i32]),
    "ag_mat2_compose": (i32, [vp, vp, vp, i32, vp]),
    "ag_lafs_left_multiply": (i32, [vp, vp, vp, i32, vp]),
    "ag_affnet_forward_raw": (i32, [vp, vp, i32, vp, vp, sz, vp]),
    "ag_orinet_forward_raw": (i32, [vp, vp, i32, vp, vp, sz, vp]),
    "ag_debug_fuse_l3": (i32, [i32]),
    "ag_debug_tcx_layer": (i32, [vp, vp, i32, i32, vp, vp, sz, vp]),
    "ag_affnet_forward": (i32, [vp, vp, i32, vp, i32, vp, vp, sz, vp]),
    "ag_orinet_forward": (i32, [vp, vp, i32, vp, i32, vp, vp, vp, sz, vp]),
    "ag_hardnet_forward": (i32, [vp, vp, i32, vp, i32, vp, vp, sz, vp]),
    "ag_net_forward_pyr": (i32, [vp, C.POINTER(PyramidPlan), vp, vp, vp, vp, vp, i32, vp, vp, sz, vp]),
    "ag_affine_shape_filter": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]),
    "ag_lafs_apply_rotation": (i32, [vp, vp, i32, vp]),
    "ag_lafs_scale": (i32, [vp, vp, i32, f32, f32, f32, vp]),
    "ag_lafs_to_ell": (i32, [vp, i32, vp, vp]),
    "ag_circular_gauss_kernel": (i32, [i32, f64, vp]),
    "ag_orientation_hist": (i32, [vp, i32, i32, vp, vp, vp]),
    "ag_baumberg_shape": (i32, [vp, i32, i32, vp, vp, vp]),
    "ag_orientation_hist_pyr": (i32, [C.POINTER(PyramidPlan), vp, vp, vp, vp, vp, i32, i32, vp, vp, vp]),
    "ag_baumberg_shape_pyr": (i32, [C.POINTER(PyramidPlan), vp, vp, vp, vp, vp, i32, i32, i32, vp, vp]),
    "ag_distance_matrix": (i32, [vp, i32, vp, i32, i32, vp, vp]),
    "ag_match_snn_workspace_bytes": (sz, [i32, i32]),
    "ag_match_snn": (i32, [vp, i32, vp, i32, i32, f32, vp, sz, vp, vp, vp, vp, vp]),
    "ag_pipeline_create": (i32, [C.POINTER(PipelineConfig), vp, vp, vp, C.POINTER(vp)]),
    "ag_pipeline_create_ex": (i32, [C.POINTER(PipelineConfig), C.POINTER(PipelineEstimators), vp, vp, vp, C.POINTER(vp)]),
    "ag_pipeline_destroy": (None, [vp]),
    "ag_pipeline_workspace_bytes": (sz, [vp]),
    "ag_pipeline_plan": (C.POINTER(PyramidPlan), [vp]),
    "ag_pipeline_run": (i32, [vp, vp, vp, sz, vp, vp, vp, vp, vp]),
    "ag_pipeline_launch_count": (i32, [vp]),
}

_lib = None


def build(verbose=False):
    """Compile the CUDA sources for sm_100a into affnet_b200/lib (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["bash", os.path.join(HERE, "csrc", "build.sh")], capture_output=True, text=True)
    if r.returncode != 0:
        raise AffnetB200Error("building libaffnet_b200.so failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout.strip())
    return LIB_PATH


def lib():
    """The loaded shared library with typed prototypes.  Raises if it is missing (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise AffnetB200Error("%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                  "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError => the .so is stale w.r.t. the header
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise AffnetB200Error("libaffnet_b200 error %d: %s" % (rc, lib().ag_last_error().decode()))


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())


def require_cuda(t, name="tensor"):
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise AffnetB200Error("%s must be a CUDA tensor: affnet_b200 has no CPU path" % name)
    return t


def f32c(t, name="tensor"):
    require_cuda(t, name)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def make_plan(B, H, W, nlevels=3, init_sigma=1.6, border=5):
    plan = PyramidPlan()
    check(lib().ag_pyramid_plan(B, H, W, nlevels, float(init_sigma), border, C.byref(plan)))
    return plan


def profile(fn):
    """Run fn() with the per-launch event profiler on; returns [(kernel name, ms), ...] in launch order."""
    check(lib().ag_prof_begin(stream_ptr()))
    try:
        fn()
    finally:
        n = lib().ag_prof_end()
    if n < 0:
        check(n)
    out = []
    for i in range(n):
        name, ms = C.c_char_p(), C.c_float()
        check(lib().ag_prof_get(i, C.byref(name), C.byref(ms)))
        out.append((name.value.decode(), ms.value))
    return out
