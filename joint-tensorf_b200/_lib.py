"""ctypes binding of csrc/libjt_vm.so (the C ABI declared in include/jt_vm.h).

There is no CPU fallback: if the shared library is missing or a CUDA device is
not present, every op raises. Build with `python -c "import __graft_entry__ as
g; g.build()"` or `joint-tensorf_b200/csrc/build.sh`.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libjt_vm.so")

_P, _I, _F, _D = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double

# name -> argtypes; mirrors include/jt_vm.h one to one (tests/test_abi.py checks it)
SIGNATURES = {
    "jt_sample_ray_dense": [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_march_compact": [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_exclusive_scan": [_P, _P, _I, _P],
    "jt_vm_gather_fwd": [_I, _P, _P, _P, _P, _P, _I, _P, _P],
    "jt_vm_gather_bwd": [_I, _P, _P, _P, _P, _P, _P, _I, _P, _P, _I, _P],
    "jt_vm_scatter_rays": [_I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _I, _P, _P, _P, _I, _I, _P],
    "jt_ray_init": [_P, _P, _I, _P, _P, _P],
    "jt_gemm_nt": [_P, _I, _P, _I, _I, _P, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P],
    "jt_gemm_tn": [_P, _I, _P, _I, _P, _I, _I, _I, _P, _I, _P, _P],
    "jt_pe_encode": [_I, _I, _I, _I, _I, _F, _F, _I, _I, _P, _I, _P, _P, _P, _P, _I, _P, _I, _P, _I, _P, _I, _P],
    "jt_sh_shade": [_I, _P, _I, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _I, _P],
    "jt_tc_selftest": [_I, _P, _I, _P, _I, _P, _I, _I, _I, _P],
    "jt_app_basis_fwd_tc": [_I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _I, _P, _P, _P],
    "jt_head_mlp_fwd_tc": [_I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _F, _F, _P, _P, _P],
    "jt_head_bwd_tc": [_P, _P, _I, _P, _P, _P, _P, _P, _I, _F, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_app_basis_sh_fwd_tc": [_I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _I, _P, _P, _P, _P],
    "jt_sh_bwd_tc": [_P, _P, _I, _P, _P, _I, _P, _I, _P, _P, _P],
    "jt_alpha_fwd": [_P, _I, _P, _P, _P, _F, _I, _F, _F, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P],
    "jt_composite_fwd": [_P, _I, _P, _P, _P, _P, _P, _P, _I, _F, _P, _P, _P, _P, _I, _P],
    "jt_render_bwd": [_P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _F, _I, _F, _I, _I, _P, _P, _P, _P],
    "jt_blur_cl": [_P, _P, _P, _I, _I, _I, _P, _I, _I, _I, _P],
    "jt_blur_multi": [_I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "jt_pose_rays_fwd": [_P, _P, _P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P],
    "jt_pose_rays_bwd": [_P, _P, _P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P],
    "jt_reg_values": [_I, _P, _P, _P, _P, _P, _P, _P],
    "jt_reg_grads": [_I, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_field_alpha": [_P, _P, _P, _P, ctypes.c_longlong, _P, _P, _P, _P, _P, _P, _P, _F, _I, _F, _P, _P],
    "jt_field_density_grad": [_P, _P, _P, _P, _P, _P, _P, ctypes.c_longlong, _P, _P, _P, _F, _I, _I, _P, _P, _P],
    "jt_raycast": [_P, _P, _P, _P, _P, _P, _F, _I, _F, _F, _P, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P],
    "jt_normal_composite": [_P, _I, _P, _P, _P, _P, _P, _F, _P, _P, _P, _P],
    "jt_alpha_mask_build": [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P],
    "jt_resize_bilinear_cl": [_P, _I, _I, _I, _P, _I, _I, _P],
    "jt_mc_count": [_P, _I, _I, _I, _F, _P, _P, _P],
    "jt_mc_emit": [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_mc_normals": [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_image_blur": [_P, _P, _P, _I, _I, _I, _P, _I, _P],
    "jt_edge_mask": [_P, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P],
    "jt_render_loss_fwd": [_P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _F, _F, _P, _P, _P],
    "jt_render_loss_bwd": [_P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _F, _F, _P, _P, _P, _P],
    "jt_wv_head_fwd_tc": [_P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _F, _F, _P, _P, _P, _P],
    "jt_wv_head_bwd_tc": [_P, _P, _P, _P, _P, _P, _P, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "jt_cast_bf16_multi": [_I, _P, _P, _P, _P],
    "jt_adam_multi": [_I, _P, _P, _P, _P, _P, _P, _P, _D, _D, _D, _D, _I, _P],
}

_lib = None


class JtError(RuntimeError):
    pass


def lib():
    """The loaded CDLL. Raises (loudly) when the CUDA library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise JtError(
                f"{LIB_PATH} not found: the CUDA extension is not built. There is no CPU fallback; "
                "run `python -c \"import __graft_entry__ as g; g.build()\"`.")
        cdll = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(cdll, name)
            fn.argtypes = args
            fn.restype = _I
        cdll.jt_strerror.argtypes = [_I]
        cdll.jt_strerror.restype = ctypes.c_char_p
        cdll.jt_version.argtypes = []
        cdll.jt_version.restype = _I
        cdll.jt_head_tc_stage_bytes.argtypes = [_I]
        cdll.jt_head_tc_stage_bytes.restype = ctypes.c_longlong
        cdll.jt_wv_stage_bytes.argtypes = [_I]
        cdll.jt_wv_stage_bytes.restype = ctypes.c_longlong
        cdll.jt_edge_mask_ws_floats.argtypes = [_I, _I, _I]
        cdll.jt_edge_mask_ws_floats.restype = ctypes.c_longlong
        cdll.jt_mc_scratch_bytes.argtypes = [_I, _I, _I]
        cdll.jt_mc_scratch_bytes.restype = ctypes.c_longlong
        cdll.jt_launch_count.argtypes = []
        cdll.jt_launch_count.restype = ctypes.c_longlong
        _lib = cdll
    return _lib


def check(rc, what):
    if rc != 0:
        raise JtError(f"{what} failed: {lib().jt_strerror(rc).decode()} (code {rc})")


def launch_count():
    return int(lib().jt_launch_count())


def floats(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])


def ints(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


def doubles(vals):
    return (ctypes.c_double * len(vals))(*[float(v) for v in vals])


def longlongs(vals):
    return (ctypes.c_longlong * len(vals))(*[int(v) for v in vals])


def ptrs(vals):
    return (ctypes.c_void_p * len(vals))(*[int(v) for v in vals])
