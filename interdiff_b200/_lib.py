"""ctypes binding of libinterdiff_b200.so (the C ABI in include/interdiff_b200.h).

There is NO CPU or PyTorch fallback: importing the product ops without the built library, or
calling them without a Blackwell GPU, raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libinterdiff_b200.so")


class DenoiserConfig(C.Structure):
    _fields_ = [("variant", C.c_int), ("d_model", C.c_int), ("n_heads", C.c_int), ("d_ff", C.c_int),
                ("n_layers", C.c_int), ("n_queries", C.c_int), ("c_body", C.c_int), ("c_obj", C.c_int),
                ("c_extra", C.c_int), ("n_points", C.c_int), ("qan_mask", C.c_int),
                ("rotary_offsets", C.c_float * 3)]


_P = C.c_void_p
_SIGS = {
    "idb_version": (C.c_int, []),
    "idb_create": (C.c_int, [C.POINTER(_P)]),
    "idb_destroy": (C.c_int, [_P]),
    "idb_last_error": (C.c_char_p, [_P]),
    "idb_launch_count": (C.c_longlong, [_P]),
    "idb_encode_condition": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "idb_encode_condition_skeleton": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "idb_skeleton_metrics": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "idb_pointcloud_embed": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P]),
    "idb_metrics": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "idb_rollout_next_window": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "idb_add_offset": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, _P, _P, C.c_float, _P]),
    "idb_debug_set_gemm_multicast": (C.c_int, [_P, C.c_int]),
    "idb_debug_max_layer_clusters": (C.c_int, [_P]),
    "idb_smooth": (C.c_int, [_P, C.c_int, C.c_int, C.c_longlong, _P, _P]),
    "idb_metric_min": (C.c_int, [_P, C.c_longlong, _P, _P, _P]),
    "idb_set_gemm_backend": (C.c_int, [_P, C.c_int]),
    "idb_set_dependent_launch": (C.c_int, [_P, C.c_int]),
    "idb_set_fused_mlp": (C.c_int, [_P, C.c_int]),
    "idb_set_nn_pruning": (C.c_int, [_P, C.c_int]),
    "idb_debug_mlp": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "idb_debug_last_ms": (C.c_double, [_P]),
    "idb_denoiser_init": (C.c_int, [_P, C.POINTER(DenoiserConfig)]),
    "idb_denoiser_load": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int]),
    "idb_denoiser_commit": (C.c_int, [_P]),
    "idb_denoiser_bind": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "idb_denoiser_forward": (C.c_int, [_P, _P, _P, _P, _P]),
    "idb_diffusion_init": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int]),
    "idb_p_sample": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "idb_p_sample_predict": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P]),
    "idb_p_sample_finish": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P]),
    "idb_p_sample_loop": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, _P, _P]),
    "idb_body_init": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "idb_smplh_lbs": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P]),
    "idb_vertex_normals": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "idb_signed_nn": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "idb_rot6d_to_axis_angle": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "idb_projector_init": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int]),
    "idb_projector_load": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int]),
    "idb_projector_commit": (C.c_int, [_P]),
    "idb_projector_set_hand_markers": (C.c_int, [_P, _P, C.c_int]),
    "idb_projector_sample": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "idb_correction_bind": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, C.c_int, _P]),
    "idb_debug_gemm": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "idb_debug_gemm_repeat": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "idb_debug_set_gemm_accumulators": (C.c_int, [C.c_int]),
    "idb_debug_attn_trace": (C.c_int, [C.POINTER(C.c_longlong)]),
    "idb_debug_split": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "idb_debug_gemm_presplit": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "idb_debug_chain_trace": (C.c_int, [_P, _P]),
    "idb_debug_gemm_trace": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "idb_correction_apply": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, _P, _P]),
    "idb_projector_init_skeleton": (C.c_int, [_P, C.c_int, C.c_int, C.c_int]),
    "idb_projector_sample_skeleton": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "idb_skeleton_correction_apply": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int, _P]),
    "idb_correction_set_log": (C.c_int, [_P, _P, _P, C.c_int]),
}

EXPORTS = sorted(_SIGS)
_lib = None


def lib():
    """Returns the loaded library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "interdiff_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the product path)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
