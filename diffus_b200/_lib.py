"""ctypes binding of ``libdiffus_b200.so`` (the C ABI declared in ``include/diffus_b200.h``).

There is no CPU implementation behind these symbols and no fallback: if the shared library
is missing or a symbol is absent, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdiffus_b200.so")
ABI_VERSION = 1

SAMPLER_NEAREST, SAMPLER_TRILINEAR = 0, 1
LAYOUT_LINEAR, LAYOUT_BRICK, LAYOUT_QUAD, LAYOUT_TEXTURE = 0, 1, 2, 3
POSE_F32, POSE_F64, POSE_F32_PER_RAY = 0, 1, 2
PROBE_CONVEX, PROBE_LINEAR = 0, 1
MLP_NPARAMS = 1153


class DiffusVolume(C.Structure):
    _fields_ = [("data", C.c_void_p), ("dim", C.c_int32 * 3), ("layout", C.c_int32)]


class DiffusRenderArgs(C.Structure):
    _fields_ = [
        ("volume", DiffusVolume),
        ("sources", C.c_void_p),
        ("directions", C.c_void_p),
        ("pose_dtype", C.c_int32),
        ("product_f32", C.c_int32),
        ("n_poses", C.c_int64),
        ("n_rays", C.c_int64),
        ("dir_pose_stride", C.c_int64),
        ("n_samples", C.c_int32),
        ("start", C.c_int32),
        ("sampler", C.c_int32),
        ("attenuation", C.c_float),
        ("frame", C.c_void_p),
        ("seg_prefix", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
    ]


class DiffusRenderBwdArgs(C.Structure):
    _fields_ = [
        ("fwd", DiffusRenderArgs),
        ("grad_frame", C.c_void_p),
        ("grad_volume", C.c_void_p),
        ("grad_sources", C.c_void_p),
        ("grad_directions", C.c_void_p),
        ("target", C.c_void_p),
        ("grad_scale", C.c_float),
        ("loss_scale", C.c_float),
        ("loss", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
    ]


class DiffusGaussNewtonArgs(C.Structure):
    _fields_ = [
        ("fwd", DiffusRenderArgs),
        ("target", C.c_void_p),
        ("loss", C.c_void_p),
        ("jtr", C.c_void_p),
        ("jtj", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
    ]


class DiffusGaussNewtonSweepArgs(C.Structure):
    _fields_ = [
        ("fwd", DiffusRenderArgs),
        ("target", C.c_void_p),
        ("pivot", C.c_void_p),
        ("loss", C.c_void_p),
        ("jtr", C.c_void_p),
        ("jtj", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
    ]


_P = C.POINTER
_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# symbol -> (restype, argtypes); must list every function declared in include/diffus_b200.h
SIGNATURES = {
    "diffus_abi_version": (_i32, []),
    "diffus_error_string": (C.c_char_p, [_i32]),
    "diffus_render_workspace_bytes": (_i64, [_P(DiffusRenderArgs)]),
    "diffus_render_forward": (_i32, [_P(DiffusRenderArgs), _vp]),
    "diffus_render_bwd_workspace_bytes": (_i64, [_P(DiffusRenderBwdArgs)]),
    "diffus_render_bwd_needs_prefix": (_i32, [_P(DiffusRenderBwdArgs)]),
    "diffus_render_backward": (_i32, [_P(DiffusRenderBwdArgs), _vp]),
    "diffus_render_gauss_newton_workspace_bytes": (_i64, [_P(DiffusGaussNewtonArgs)]),
    "diffus_render_gauss_newton": (_i32, [_P(DiffusGaussNewtonArgs), _vp]),
    "diffus_render_gauss_newton_sweep_workspace_bytes": (_i64, [_P(DiffusGaussNewtonSweepArgs)]),
    "diffus_render_gauss_newton_sweep": (_i32, [_P(DiffusGaussNewtonSweepArgs), _vp]),
    "diffus_ray_indices": (_i32, [_P(DiffusRenderArgs), _vp, _vp, _vp, _vp]),
    "diffus_trace_values": (_i32, [_P(DiffusRenderArgs), _vp, _vp]),
    "diffus_sample_points": (_i32, [_P(DiffusVolume), _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "diffus_trace_values_backward": (_i32, [_P(DiffusRenderArgs), _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "diffus_echo_forward": (_i32, [_vp, _i64, _i32, _vp, _vp]),
    "diffus_echo_backward": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "diffus_cone_directions": (_i32, [_vp, _i64, _i64, _f64, _vp, _vp]),
    "diffus_mlp_forward": (_i32, [_vp, _vp, _vp, _i64, _f32, _f32, _vp, _vp]),
    "diffus_mlp_forward_ex": (_i32, [_vp, _vp, _vp, _i64, _f32, _f32, _vp, _i32, _vp]),
    "diffus_mlp_bwd_workspace_bytes": (_i64, [_i64]),
    "diffus_mlp_backward": (_i32, [_vp, _vp, _vp, _vp, _i64, _f32, _vp, _vp, _i64, _vp]),
    "diffus_splat_workspace_bytes": (_i64, [_i32, _i32]),
    "diffus_splat_forward": (_i32, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _i64, _vp]),
    "diffus_splat_backward": (_i32, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _i64, _vp]),
    "diffus_mlp_backward_ex": (_i32, [_vp, _vp, _vp, _vp, _i64, _f32, _vp, _vp, _i64, _i32, _vp]),
    "diffus_mlp_input_grad": (_i32, [_vp, _vp, _vp, _vp, _i64, _f32, _vp, _vp]),
    "diffus_brain_mask": (_i32, [_vp, _P(_i32 * 3), _f32, _i32, _vp, _vp, _vp]),
    "diffus_masked_zscore": (_i32, [_vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "diffus_brick_elems": (_i64, [_P(_i32 * 3)]),
    "diffus_volume_to_bricks": (_i32, [_vp, _P(_i32 * 3), _vp, _vp]),
    "diffus_bricks_to_volume": (_i32, [_vp, _P(_i32 * 3), _vp, _vp]),
    "diffus_fan_directions": (_i32, [_vp, _vp, _i64, _i64, C.c_double, _vp, _vp]),
    "diffus_fan_directions_backward": (_i32, [_vp, _vp, _vp, _i64, _i64, C.c_double, _vp, _vp, _vp]),
    "diffus_probe_rays": (_i32, [_i32, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _f64, _vp, _vp, _vp]),
    "diffus_probe_rays_backward": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _f64, _vp, _vp, _vp, _vp]),
    "diffus_gather_probe": (_i32, [_vp, _i64, _i32, _i64, C.c_uint32, _vp, _vp]),
    "diffus_volume_texture_create": (_i32, [_vp, _P(_i32 * 3), _P(C.c_uint64), _P(C.c_uint64), _vp]),
    "diffus_volume_texture_update": (_i32, [C.c_uint64, _vp, _P(_i32 * 3), _vp]),
    "diffus_volume_texture_destroy": (_i32, [C.c_uint64, C.c_uint64]),
    "diffus_adam_step": (_i32, [_vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _vp]),
    "diffus_volume_slice": (_i32, [_vp, _P(_i32 * 3), _i32, _i32, _i32, _vp, _i32, _vp]),
    "diffus_conv1d_rows_forward": (_i32, [_vp, _i64, _i32, _vp, _i32, _i32, _vp, _vp]),
    "diffus_conv1d_rows_backward": (_i32, [_vp, _i64, _i32, _vp, _i32, _i32, _vp, _vp]),
    "diffus_rotate_around_apex": (_i32, [_vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp]),
    "diffus_log_compress_forward": (_i32, [_vp, _i64, _vp, _vp, _vp]),
    "diffus_log_compress_backward": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "diffus_rf_to_bmode": (_i32, [_vp, _i64, _i32, _vp, _vp, _vp, _i64, _vp]),
    "diffus_masked_mse_edge_forward": (_i32, [_vp, _vp, _vp, _i32, _i32, _f32, _vp, _vp]),
    "diffus_masked_mse_edge_backward": (_i32, [_vp, _vp, _vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp]),
    "diffus_ssim_workspace_bytes": (_i64, [_i32, _i32, _i32]),
    "diffus_ssim_loss_forward": (_i32, [_vp, _vp, _i32, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _i64, _vp]),
    "diffus_ssim_loss_backward": (_i32, [_vp, _vp, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _i64, _vp]),
    "diffus_quad_elems": (_i64, [_P(_i32 * 3)]),
    "diffus_volume_to_quads": (_i32, [_vp, _P(_i32 * 3), _vp, _vp]),
    "diffus_volume_gaussian_blur": (_i32, [_vp, _P(_i32 * 3), _f32, _f32, _vp, _vp, _vp]),
}

_lib = None


class DiffusError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built -- no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DIFFUS_B200_LIB", LIB_PATH)     # development aid: point at another build of the same ABI
    if not os.path.exists(path):
        raise DiffusError(
            f"{path} not found: the CUDA library has not been built. "
            "Run `python -m diffus_b200.build` (or `__graft_entry__.build()`); there is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    got = lib.diffus_abi_version()
    if got != ABI_VERSION:
        raise DiffusError(f"ABI mismatch: library {got}, binding {ABI_VERSION}; rebuild the library")
    _lib = lib
    return lib


def check(code: int, what: str):
    if code != 0:
        msg = load().diffus_error_string(code).decode()
        raise DiffusError(f"{what} failed with code {code}: {msg}")


def check_count(code: int, what: str) -> int:
    """For entry points that answer with a non-negative number (negative = error code)."""
    if code < 0:
        check(code, what)
    return code
