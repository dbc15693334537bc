"""ctypes binding of libvsr_b200.so (include/vsr_b200.h).  There is no fallback: if the library is
missing the import fails, and every op raises on non-CUDA tensors."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvsr_b200.so")

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_i64 = ctypes.c_int64
c_size_t = ctypes.c_size_t
c_float = ctypes.c_float


class VsrError(RuntimeError):
    pass


class SrfbnConfig(ctypes.Structure):
    _fields_ = [("num_maps", ctypes.c_int32), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
                ("num_steps", ctypes.c_int32), ("num_groups", ctypes.c_int32),
                ("num_features", ctypes.c_int32), ("upscale", ctypes.c_int32)]


_fp = ctypes.POINTER(c_float)


class SrfbnWeights(ctypes.Structure):
    _fields_ = [
        ("sub_mean_bias", _fp), ("add_mean_bias", _fp),
        ("conv_in_w", _fp), ("conv_in_b", _fp), ("conv_in_slope", c_float),
        ("feat_in_w", _fp), ("feat_in_b", _fp), ("feat_in_slope", c_float),
        ("compress_in_w", _fp), ("compress_in_b", _fp), ("compress_in_slope", c_float),
        ("up_w", _fp * 6), ("up_b", _fp * 6), ("up_slope", c_float * 6),
        ("down_w", _fp * 6), ("down_b", _fp * 6), ("down_slope", c_float * 6),
        ("uptran_w", _fp * 5), ("uptran_b", _fp * 5), ("uptran_slope", c_float * 5),
        ("downtran_w", _fp * 5), ("downtran_b", _fp * 5), ("downtran_slope", c_float * 5),
        ("compress_out_w", _fp), ("compress_out_b", _fp), ("compress_out_slope", c_float),
        ("out_w", _fp), ("out_b", _fp), ("out_slope", c_float),
        ("conv_out_w", _fp), ("conv_out_b", _fp),
        ("fc0_w", _fp), ("fc0_b", _fp), ("fc2_w", _fp), ("fc2_b", _fp),
    ]


# name -> (restype, argtypes); mirrors include/vsr_b200.h one to one
SIGNATURES = {
    "vsr_version": (ctypes.c_char_p, []),
    "vsr_launch_count": (ctypes.c_uint64, []),
    "vsr_launch_count_reset": (None, []),
    "vsr_error_string": (ctypes.c_char_p, [c_int]),
    "vsr_resample2d_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vsr_warp_nhwc_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vsr_warp_windows_nhwc3": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p] + [c_int] * 6 + [c_void_p]),
    "vsr_compose_flow_windows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_i64, c_int, c_int, c_void_p]),
    "vsr_warp_labels_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vsr_warp_labels_u8_windows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_i64, c_int, c_int, c_void_p]),
    "vsr_channelnorm_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vsr_channelnorm_forward_typed": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vsr_channelnorm_backward_typed": (c_int, [c_void_p] * 4 + [c_int] * 6 + [c_void_p]),
    "vsr_resample2d_backward": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p]),
    "vsr_channelnorm_backward": (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p]),
    "vsr_resample2d_backward_deterministic_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "vsr_resample2d_backward_deterministic": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p, c_size_t, c_void_p]),
    "vsr_correlation_output_shape": (c_int, [c_int] * 8 + [ctypes.POINTER(c_int)] * 3),
    "vsr_correlation_forward": (c_int, [c_void_p] * 3 + [c_int] * 10 + [c_void_p]),
    "vsr_correlation_backward": (c_int, [c_void_p] * 5 + [c_int] * 10 + [c_void_p]),
    "vsr_flow_projection_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "vsr_flow_projection_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "vsr_flow_projection_forward_bounded": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_float, c_void_p]),
    "vsr_flow_projection_deterministic_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "vsr_flow_projection_forward_deterministic": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "vsr_vos_threshold_windows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vsr_flow_to_image": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "vsr_mask_fill": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vsr_assemble_stack_windows": (c_int, [c_void_p] * 8 + [c_int, c_i64, c_int, c_int, c_int, c_int, c_void_p]),
    "vsr_estimate_slot_windows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_i64, c_int, c_int, c_int, c_void_p]),
    "vsr_srfbn_plan_create": (c_int, [ctypes.POINTER(SrfbnConfig), ctypes.POINTER(c_void_p)]),
    "vsr_srfbn_plan_destroy": (None, [c_void_p]),
    "vsr_srfbn_plan_set_workspace_cap": (c_int, [c_void_p, c_size_t]),
    "vsr_srfbn_chunk_maps": (c_int, [c_void_p]),
    "vsr_srfbn_plan_set_windows": (c_int, [c_void_p, c_int]),
    "vsr_srfbn_weight_bytes": (c_size_t, [c_void_p]),
    "vsr_srfbn_workspace_bytes": (c_size_t, [c_void_p]),
    "vsr_srfbn_pack_weights": (c_int, [c_void_p, ctypes.POINTER(SrfbnWeights), c_void_p]),
    "vsr_srfbn_bind": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    "vsr_srfbn_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "vsr_srfbn_forward_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vsr_srfbn_prepare_refresh": (c_int, [c_void_p, c_int]),
    "vsr_srfbn_forward_refresh_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "vsr_srfbn_plan_set_map_range": (c_int, [c_void_p, c_int, c_int]),
    "vsr_srfbn_forward_maps": (c_int, [c_void_p, c_void_p, c_void_p]),
    "vsr_srfbn_forward_maps_refresh": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "vsr_srfbn_pack_bands": (c_int, [c_void_p, ctypes.POINTER(c_int), c_int, c_void_p, c_void_p]),
    "vsr_srfbn_fuse_band": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "vsr_unpack_bands": (c_int, [c_void_p, c_void_p, c_int, c_i64, c_i64, ctypes.POINTER(c_int), c_int, c_i64,
                                 c_void_p]),
    "vsr_srfbn_kernel_class_name":(ctypes.c_char_p, [c_int]),
    "vsr_srfbn_profile_enable": (c_int, [c_void_p, c_int]),
    "vsr_srfbn_profile_read": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vsr_srfbn_profile_launches": (c_int, [c_void_p, c_void_p, c_void_p, c_int]),
    "vsr_srfbn_debug_premix": (c_int, [c_void_p, c_void_p, c_void_p]),
    "vsr_test_pointwise": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_float, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsr_test_deconv": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsr_test_fused_down": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                    c_float, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsr_test_fused_updown": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float,
                                      c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                      c_size_t, c_void_p]),
    "vsr_test_x2_layer": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_size_t, c_void_p]),
    "vsr_test_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m video_super_resolution_b200.build` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().vsr_error_string(code).decode()
        raise VsrError(f"{what}: {msg} (code {code})" if what else f"{msg} (code {code})")


def launch_count() -> int:
    return int(lib().vsr_launch_count())


def launch_count_reset() -> None:
    lib().vsr_launch_count_reset()
