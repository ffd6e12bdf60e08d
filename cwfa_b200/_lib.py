"""ctypes binding of the C-ABI library (include/cwfa_b200.h).

There is NO CPU fallback: if the shared library cannot be built/loaded the import of the
compute path fails loudly, and every op refuses non-CUDA tensors.
"""
import ctypes as C
import os
import threading

from . import _build

_lock = threading.Lock()
_lib = None

i32, i64, f32, f64, vp = C.c_int, C.c_int64, C.c_float, C.c_double, C.c_void_p

# name -> argtypes (restype is int unless listed in _RESTYPES)
_SIGS = {
    "cwfa_device_check": [],
    "cwfa_haar1d_fwd": [vp, vp, vp, i32, i32, i64, i64, i64, vp],
    "cwfa_haar1d_inv": [vp, vp, vp, i32, i32, i64, i64, i64, vp],
    "cwfa_haar2d_down": [vp, vp, i32, i32, i32, i32, i32, f32, vp],
    "cwfa_haar2d_up": [vp, vp, i32, i32, i32, i32, i32, f32, vp],
    "cwfa_permute": [vp, vp, vp, i32, i32, i32, i32, i32, vp],
    "cwfa_affine_workspace_blocks": [],
    "cwfa_affine": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i64, i64, i64, f32, f32, f32, i32, vp],
    "cwfa_conv2d_f32": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_convT2x2_f32": [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
    "cwfa_depth_stencil3d_f32": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
    "cwfa_stats_workspace_blocks": [],
    "cwfa_channel_stats_f32": [vp, vp, vp, i32, i32, i64, vp],
    "cwfa_bn_finalize_f32": [vp, vp, vp, vp, vp, i32, f64, f32, vp],
    "cwfa_scale_shift_f32": [vp, vp, vp, vp, i32, i32, i64, vp],
    "cwfa_maxpool2_f32": [vp, vp, i32, i32, i32, i32, vp],
    "cwfa_layernorm_workspace_blocks": [],
    "cwfa_layernorm_chw_f32": [vp, vp, vp, vp, vp, i32, i64, f32, vp],
    "cwfa_gate_add_f32": [vp, vp, vp, i64, vp],
    "cwfa_cast_f32_f16": [vp, vp, i64, vp],
    "cwfa_extract_views": [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, f32, f32, i32, vp],
    "cwfa_extract_views_c8": [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, f32, i32, i32, vp],
    "cwfa_attention_gate_f32": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i64, vp],
    "cwfa_tc_kc": [i32],
    "cwfa_tc_pack_weights": [vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_conv_tc": [vp, vp, vp, vp, vp, vp] + [i32] * 14 + [vp],
    "cwfa_conv_tc_plan": [i32] * 17 + [vp],
    "cwfa_conv_tc_bn": [vp, vp, vp, vp, vp] + [i32] * 12 + [vp, vp],
    "cwfa_bn_partial_finalize": [vp, i32, i32, i32, i32, i32, vp, vp, f32, vp, vp, vp, vp],
    "cwfa_resblock_tc": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_c8_stats_workspace_floats": [i32],
    "cwfa_c8_prelu": [vp, vp, vp, i32, i32, i64, i32, vp],
    "cwfa_c8_prelu_bwd": [vp, vp, vp, vp, vp, vp, i32, i32, i64, i32, vp],
    "cwfa_c8_elu_bwd": [vp, vp, vp, vp, vp, i32, i32, i64, i32, vp],
    "cwfa_c8_channel_stats": [vp, vp, vp, i32, i32, i64, i32, vp],
    "cwfa_c8_bn_batch_scale_shift": [vp, vp, vp, f32, vp, vp, vp, i32, i32, i64, i32, vp],
    "cwfa_c8_bn_apply": [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
    "cwfa_c8_col2im3x3": [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_stencil3d_tc": [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_c8_layernorm_workspace_floats": [i32],
    "cwfa_c8_layernorm": [vp, vp, vp, vp, vp, i32, i32, i32, i64, f32, i32, vp],
    "cwfa_conv_tc_coupling_tiles": [i32, i32, i32],
    "cwfa_conv_tc_coupling": [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, f32, vp, i32, i32, f32, f32,
                              i32, vp, i32, vp],
    "cwfa_coupling_tc_tiles": [i32, i32],
    "cwfa_coupling_tc": [vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, f32, vp, i32, i32, f32, f32, i32, vp, vp, vp, i32, vp, i32, i32, i32, vp],
    "cwfa_resblock_tc_batched": [vp, vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, i32, i32, vp],
    "cwfa_coupling_finalize": [vp, vp, vp, i32, i32, i32, vp],
    "cwfa_coupling_f8": [vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, f32, vp, i32, f32, f32, i32, vp, vp, vp, i32, vp, i32, i32, i32, vp],
    "cwfa_coupling_f8_samples": [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, f32, vp, i32, f32, f32, i32, vp, vp, vp, i32, vp,
                                 i32, i32, i32, vp],
    "cwfa_coupling_f8_map": [vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, f32, vp, i32, f32, f32, i32, vp, vp, vp, i32, vp, i32, i32, i32,
                             vp, vp, vp, vp, i32],
    "cwfa_haar1d_inv_stats": [vp, i32, vp, i32, vp, vp, i32, i32, i64, vp],
    "cwfa_haar1d_fwd_f8": [vp, vp, vp, i32, i32, i64, vp],
    "cwfa_haar1d_inv_f8": [vp, vp, vp, i32, i32, i64, vp],
    "cwfa_nchw_to_f8": [vp, vp, vp, i32, i32, i64, vp],
    "cwfa_f8_to_nchw": [vp, vp, vp, i32, i32, i64, vp],
    "cwfa_nchw_to_c8": [vp, vp, i32, i32, i32, i64, i32, vp],
    "cwfa_c8_to_nchw": [vp, vp, i32, i32, i32, i64, i32, vp],
    # training-time adjoints (csrc/backward.cu)
    "cwfa_conv2d_wgrad_f32": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_conv2d_dgrad_weights_f32": [vp, vp, i32, i32, i32, i32, vp],
    "cwfa_wgrad_tc": [vp, vp, vp, vp] + [i32] * 10 + [vp],
    "cwfa_elu_bwd_f32": [vp, vp, vp, i64, vp],
    "cwfa_dy_prep_workspace_floats": [i32, i32],
    "cwfa_dy_prep": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, vp],
    "cwfa_axpby_f32": [vp, vp, vp, f32, f32, i64, vp],
    "cwfa_prelu_f32": [vp, vp, vp, i64, vp],
    "cwfa_reduce_workspace_blocks": [],
    "cwfa_prelu_bwd_f32": [vp, vp, vp, vp, vp, vp, i64, vp],
    "cwfa_affine_bwd": [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i64, i64, i64, i64, i64, f32, f32, f32, i32, vp],
    "cwfa_stencil3d_1toC_f32": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_stencil3d_Cto1_f32": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_stencil3d_wgrad_workspace_floats": [i32],
    "cwfa_stencil3d_wgrad_f32": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp],
    "cwfa_lion_step_f32": [vp, vp, vp, i64, f32, f32, f32, f32, f32, vp],
    "cwfa_lion_step_masked_f32": [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, vp],
    "cwfa_act_bwd_f32": [vp, vp, vp, i64, i32, vp],
    "cwfa_gelu_add_f32": [vp, vp, vp, vp, i64, vp],
    "cwfa_ln_bwd_stats_f32": [vp, vp, vp, vp, vp, i32, i64, vp],
    "cwfa_ln_bwd_apply_f32": [vp, vp, vp, vp, vp, vp, vp, i32, i64, vp],
    "cwfa_gate_f32": [vp, vp, vp, vp, vp, vp, i64, vp],
    "cwfa_channel_dot_workspace_blocks": [],
    "cwfa_channel_dot_stats_f32": [vp, vp, vp, vp, i32, i32, i64, vp],
    "cwfa_bn_bwd_apply_f32": [vp, vp, vp, vp, vp, vp, i32, i32, i64, vp],
    "cwfa_maxpool2_bwd_f32": [vp, vp, vp, i32, i32, i32, i32, vp],
    "cwfa_pixel_shuffle2_f32": [vp, vp, vp, i32, i32, i32, i32, i32, vp],
}
_I64_FUNCS = {"cwfa_tc_packed_weight_elems": [i32, i32, i32, i32, i32],
              "cwfa_conv_tc_stats_floats": [i32, i32, i32, i32, i32],
              "cwfa_conv2d_wgrad_workspace_floats": [i32] * 7,
              "cwfa_wgrad_tc_workspace_floats": [i32] * 8}
_RESTYPES = {"cwfa_version": C.c_char_p, "cwfa_last_error": C.c_char_p}
# private profiling hooks (csrc/cwfa_b200_debug.h): bound for scripts/trace_*.py, not part of the public header
_OPTIONAL = {"cwfa_tc_set_debug_buffer": [vp], "cwfa_resblock_set_debug_buffer": [vp], "cwfa_stencil_set_debug_buffer": [vp]}


def exported_symbols():
    """Every symbol include/cwfa_b200.h declares (used by the CPU-side ABI test)."""
    return sorted(list(_SIGS) + list(_RESTYPES) + list(_I64_FUNCS))


def lib_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (building first if the .so is missing or stale and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        try:
            path = _build.build()
        except Exception as e:
            # A library that does not match the sources must never be bound with this file's argtypes (raw device
            # pointers through a mismatched ABI = silent memory corruption): refuse it.
            if os.path.exists(path) and _build.built_hash() == _build.source_hash():
                pass                     # up to date; the failure was incidental (e.g. nvcc absent on a deploy box)
            else:
                raise RuntimeError(
                    "cwfa_b200: the CUDA library is missing or older than its sources and could not be (re)built "
                    f"({e}); there is no CPU fallback") from e
        lib = C.CDLL(path)
        for name, args in {**_SIGS, **_OPTIONAL}.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int
        for name, args in _I64_FUNCS.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int64
        for name, rt in _RESTYPES.items():
            fn = getattr(lib, name)
            fn.argtypes = []
            fn.restype = rt
        _lib = lib
    return _lib


class CwfaError(RuntimeError):
    pass


# kernel launches issued per C-ABI call (for bench.py's "gpu_launches" claim)
_LAUNCHES = {"cwfa_bn_partial_finalize": 2, "cwfa_affine": 2, "cwfa_channel_stats_f32": 2, "cwfa_layernorm_chw_f32": 2, "cwfa_c8_channel_stats": 2, "cwfa_c8_layernorm": 2, "cwfa_conv2d_wgrad_f32": 2, "cwfa_wgrad_tc": 2, "cwfa_prelu_bwd_f32": 2, "cwfa_stencil3d_wgrad_f32": 2,
             "cwfa_reduce_workspace_blocks": 0, "cwfa_channel_dot_workspace_blocks": 0, "cwfa_channel_dot_stats_f32": 2, "cwfa_ln_bwd_stats_f32": 2, "cwfa_stencil3d_wgrad_workspace_floats": 0,
             "cwfa_tc_set_debug_buffer": 0, "cwfa_resblock_set_debug_buffer": 0, "cwfa_device_check": 0, "cwfa_conv_tc_coupling_tiles": 0, "cwfa_coupling_tc_tiles": 0, "cwfa_conv_tc_plan": 0}
launch_count = 0
launch_hist = {}


def call(name: str, *args) -> None:
    global launch_count
    lib = load()
    rc = getattr(lib, name)(*args)
    k = _LAUNCHES.get(name, 1)
    launch_count += k
    if k:
        launch_hist[name] = launch_hist.get(name, 0) + k
    if rc != 0:
        msg = lib.cwfa_last_error().decode(errors="replace")
        raise CwfaError(f"{name} failed (code {rc}): {msg}")
