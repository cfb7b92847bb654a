"""ctypes binding of the C ABI in include/rgbd_b200.h (csrc/librgbd_b200.so).

There is no fallback: if the library is missing or fails to load, every op raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librgbd_b200.so")

ABI_VERSION = 4          # RGBD_ABI_VERSION of include/rgbd_b200.h this binding was written against

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)
c_void_pp = C.POINTER(C.c_void_p)


class ConvGemmDesc(C.Structure):
    """Mirror of ``rgbd_conv_gemm_desc``."""
    _fields_ = [
        ("a", C.c_void_p), ("a_c", C.c_int), ("a_x", C.c_int), ("a_y", C.c_int), ("a_planes", C.c_int),
        ("plane_per_img", C.c_int),
        ("w", C.c_void_p), ("slices", C.c_void_p), ("n_slices", C.c_int), ("kb_elems", C.c_int),
        ("n_img", C.c_int), ("out_h", C.c_int), ("out_w", C.c_int), ("bx", C.c_int), ("by", C.c_int),
        ("n", C.c_int), ("n_pad", C.c_int), ("block_n", C.c_int),
        ("tile_order", C.c_int), ("epi_mode", C.c_int), ("act", C.c_int),
        ("scale", C.c_void_p), ("shift", C.c_void_p), ("variant", C.c_void_p), ("gate", C.c_void_p),
        ("out", C.c_void_p), ("residual", C.c_void_p), ("pool", C.c_void_p),
        ("cells_y", C.c_int), ("cells_x", C.c_int), ("conv3x3_reuse", C.c_int),
        ("codes", C.c_void_p), ("in_h", C.c_int), ("in_w", C.c_int), ("m3_py", C.c_int), ("m3_px", C.c_int),
        ("m3_stride", C.c_int), ("m3_masked_segs", C.c_int), ("m3_n_seg", C.c_int),
        ("dsam_masked", C.c_int),
        ("next_operand", C.c_void_p), ("next_codes", C.c_void_p),
        ("next_c_pad", C.c_int), ("next_n_seg", C.c_int), ("next_masked_segs", C.c_int),
        ("pool_sq", C.c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/rgbd_b200.h declares
SIGNATURES = {
    "rgbd_abi_version": (C.c_int, []),
    "rgbd_last_error": (C.c_char_p, []),
    "rgbd_dggm_fwd": (C.c_int, [C.c_int, c_void_pp, c_void_pp, c_void_pp, c_int_p, c_int_p, c_int_p, c_void_pp, c_void_pp,
                                C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_void_p]),
    "rgbd_dggm_bwd_params": (C.c_int, [C.c_int, c_void_pp, c_int_p, c_int_p, c_int_p, c_void_pp, c_void_pp, c_void_pp,
                                       c_void_pp, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p]),
    "rgbd_gradient_features_workspace_bytes": (C.c_size_t, [C.c_int]),
    "rgbd_gradient_features": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p,
                                         C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "rgbd_pack_pixel_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                         C.c_double, c_float_p, c_float_p, C.c_float, C.c_void_p, C.c_void_p]),
    "rgbd_depth_decompose_workspace_bytes": (C.c_size_t, [C.c_int]),
    "rgbd_depth_decompose": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, c_int_p,
                                       c_int_p, c_void_pp, C.c_void_p, C.c_void_p]),
    "rgbd_dsam_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_group_norm_inplace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                          C.c_void_p]),
    "rgbd_ratio_stem_pack": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p]),
    "rgbd_conv_gemm": (C.c_int, [C.POINTER(ConvGemmDesc), C.c_void_p]),
    "rgbd_cast_bf16_pitched": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_dsam_pack_t": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_dsam_dbias": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_dsam_wgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_ratio_chain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_ratio_front": (C.c_int, [C.c_void_p] * 10 + [C.c_int] * 6 + [C.c_void_p]),
    "rgbd_ratio_stem_compact_width": (C.c_int, [C.c_int]),
    "rgbd_ratio_stem_pack_compact": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_void_p]),
    "rgbd_depth_helper_workspace_bytes": (C.c_size_t, [C.c_int]),
    "rgbd_to_grayscale": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p,
                                    C.c_void_p]),
    "rgbd_depth_select_modes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "rgbd_depth_region_codes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "rgbd_resize_workspace_bytes": (C.c_size_t, [C.c_int] * 6),
    "rgbd_resize_pil_bilinear_u8": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p]),
    "rgbd_resize_cv_linear_u8": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p, C.c_void_p]),
    "rgbd_ratio_from_features": (C.c_int, [C.c_int, c_void_pp, c_int_p, c_int_p, C.c_int, c_void_pp, c_void_pp, C.c_float, C.c_float,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "rgbd_postprocess_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "rgbd_postprocess_instances": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_float] + [C.c_void_p] * 8),
    "rgbd_label_map_rle_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "rgbd_label_map_rle": (C.c_int, [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p] * 6),
    "rgbd_instance_rle_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "rgbd_instance_rle_capacity": (C.c_size_t, [C.c_int] * 4),
    "rgbd_instance_rle": (C.c_int, [C.c_void_p] * 2 + [C.c_int] * 4 + [C.c_void_p] * 6),
    "rgbd_mask_iou": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p]),
    "rgbd_ratio_tail": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, c_void_pp, c_void_pp,
                                  C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "rgbd_adaptive_avg_pool4": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rgbd_ratio_tail_prepare": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "rgbd_ratio_tail_mlp_fx": (C.c_int, [C.c_void_p, c_void_pp, c_void_pp, C.c_float, C.c_float, C.c_void_p, C.c_int, C.c_void_p]),
    "rgbd_ratio_tail_train": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_float, C.c_float, C.c_void_p, C.c_void_p, c_void_pp, c_void_pp, C.c_void_p,
                                        C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p]),
    "rgbd_msda_fwd": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 6 + [C.c_void_p]),
    "rgbd_attention_mask": (C.c_int, [C.c_void_p] + [C.c_int] * 8 + [C.c_void_p, C.c_void_p]),
    "rgbd_masked_cross_attention": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 5 + [C.c_void_p]),
    "rgbd_layer_norm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.c_float,
                                  C.c_void_p]),
    "rgbd_window_attention_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "rgbd_window_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
}

_lib: Optional[C.CDLL] = None


class RgbdB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load librgbd_b200.so (built by ``build.py`` / ``__graft_entry__.build()``).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RgbdB200Error(
            f"{LIB_PATH} is missing: build it with `python rgb-d-instance-segmentation_b200/build.py` "
            "(rgbd_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.rgbd_abi_version() != ABI_VERSION:
        raise RgbdB200Error(f"ABI version mismatch: library reports {lib.rgbd_abi_version()}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().rgbd_last_error().decode("utf-8", "replace")
        raise RgbdB200Error(f"{what} failed (code {rc}): {msg}")


def ptr_array(ptrs) -> "C.Array":
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def int_array(vals) -> "C.Array":
    return (C.c_int * len(vals))(*[int(v) for v in vals])
