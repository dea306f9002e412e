"""ctypes binding of libgeoformer_sm100.so (the C ABI declared in include/geoformer_b200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgeoformer_sm100.so")

P, I, L, F = c_void_p, c_int, c_int64, c_float

# name -> (restype, argtypes); mirrors include/geoformer_b200.h one to one
SIGNATURES = {
    "gf_abi_version": (I, []),
    "gf_last_error": (c_char_p, []),
    "gf_init": (I, [I]),
    "gf_launch_count": (L, []),
    "gf_linear_tf32": (I, [P, P, P, P, L, I, I, I, I, I, P, P, I, P, P, P, P, P]),
    "gf_linear_ref": (I, [P, P, P, P, L, I, I, I, I, I, P, P, I, P, P, P, P, P]),
    "gf_conv3x3_f16": (I, [P, P, P, P, P, I, I, I, I, I, I, I, P]),
    "gf_conv_f16": (I, [P, P, P, P, P, I, I, I, I, I, I, I, I, I, P]),
    "gf_stem_conv7x7_f16": (I, [P, P, P, P, I, I, I, P]),
    "gf_upsample_add_f16": (I, [P, P, P, I, I, I, I, I, I, P]),
    "gf_conv_ref": (I, [P, P, P, P, P, I, I, I, I, I, I, I, I, P]),
    "gf_upsample_add_ref": (I, [P, P, P, I, I, I, I, I, I, P]),
    "gf_add_posenc": (I, [P, P, P, I, L, I, P]),
    "gf_linattn_partial_floats": (L, [I, I, I, I]),
    "gf_linear_mixed": (I, [P, P, P, P, I, I, L, I, I, I, I, I, P, P, I, P, P, P, P, P]),
    "gf_fine_layer": (I, [P, P, P, P, P, P, P, P, L, P]),
    "gf_linattn_reduce_f16": (I, [P, I, P, I, I, I, I, I, P, P, P, P]),
    "gf_linattn_apply_f16": (I, [P, I, P, P, P, I, I, I, I, I, P]),
    "gf_linattn_window_f16": (I, [P, I, P, I, P, I, P, L, I, I, I, P]),
    "gf_linattn_reduce": (I, [P, I, P, I, I, I, I, I, P, P, P, P]),
    "gf_linattn_apply": (I, [P, I, P, P, P, I, I, I, I, I, P]),
    "gf_linattn_window": (I, [P, I, P, I, P, I, P, L, I, I, I, P]),
    "gf_full_attention": (I, [P, I, P, I, P, I, P, I, I, I, I, I, P]),
    "gf_dense_kv_h16": (I, [P, I, P, I, I, I, I, I, I, P, P, P, P]),
    "gf_full_attention_tc": (I, [P, I, P, P, P, P, I, I, I, I, I, I, P]),
    "gf_full_attention_window": (I, [P, I, P, I, P, I, P, L, I, I, I, P]),
    "gf_full_attention_window_f16": (I, [P, I, P, I, P, I, P, L, I, I, I, P]),
    "gf_pack_split_f16": (I, [P, P, L, I, F, I, P]),
    "gf_similarity_f16x3": (I, [P, P, P, I, I, I, I, F, P]),
    "gf_similarity_ref": (I, [P, P, P, I, I, I, I, F, F, P]),
    "gf_dual_softmax_workspace_floats": (L, [I, I, I]),
    "gf_dual_softmax_stats": (I, [P, I, I, I, P, P, P, P, P, P]),
    "gf_dual_softmax_conf": (I, [P, I, I, I, P, P, P, P, P, P, P]),
    "gf_conf_row_col_max": (I, [P, I, I, I, P, P, P]),
    "gf_mnn_select": (I, [P, I, I, I, F, I, I, I, I, I, P, P, P, P, P]),
    "gf_coarse_match_fused_workspace_bytes": (L, [I, I, I]),
    "gf_coarse_match_fused": (I, [P, P, I, I, I, I, F, F, I, I, I, I, I, P, P, P, P]),
    "gf_coarse_match_fused_pass": (I, [P, P, I, I, I, I, F, P, I, P]),
    "gf_compact_coarse": (I, [P, P, I, I, I, I, F, P, P, P, P, P, P, P, P, L, P]),
    "gf_geo_window_table": (I, [P, P, I, I, I, I, I, I, I, I, P, P]),
    "gf_geo_self_attention": (I, [P, I, P, I, P, I, P, I, I, I, I, P, P, I, P]),
    "gf_gather_anchor_kv": (I, [P, I, P, I, I, I, I, I, P, P, I, I, P, P, P]),
    "gf_gather_anchor_kv_f16": (I, [P, I, P, I, P, I, I, I, I, I, P, P, I, I, P, P, P, P]),
    "gf_geo_self_attention_tc": (I, [P, I, P, P, P, I, I, I, I, I, P, P]),
    "gf_gather_anchor_kv_h16": (I, [P, I, P, I, I, I, I, I, P, P, I, I, P, P, P]),
    "gf_masked_softmax_rows": (I, [P, I, I, I, I, P, P]),
    "gf_gemm_tf32_batched": (I, [P, L, L, P, L, L, P, L, L, I, I, I, I, F, P]),
    "gf_geo_cross_attention": (I, [P, I, P, I, P, I, P, I, I, I, I, I, P, I, P]),
    "gf_geo_cross_attention_f16": (I, [P, I, P, I, P, I, P, I, I, I, I, I, P, I, P]),
    "gf_select_rows": (I, [P, P, P, I, L, I, P]),
    "gf_fine_gather": (I, [P, I, I, I, P, P, L, I, I, I, P, P]),
    "gf_fine_gather_f16": (I, [P, I, I, I, P, P, L, I, I, I, P, P]),
    "gf_fine_gather_f16_f16": (I, [P, I, I, I, P, P, L, I, I, I, P, P]),
    "gf_gather_rows": (I, [P, L, I, P, P, L, P, P]),
    "gf_fine_match": (I, [P, P, L, I, I, F, F, P, P, P, P, P, P]),
    "gf_resize_gray_u8": (I, [P, I, I, P, I, I, P]),
    "gf_ransac_workspace_bytes": (L, [I, I]),
    "gf_ransac_homography": (I, [P, P, P, P, L, I, I, F, ctypes.c_uint, I, I, I, I, I, P, P, P, P, P, P, P, P, P, P, P, I, P]),
    "gf_compact_fine": (I, [P, P, P, P, P, P, P, L, I, F, F, F, P, P, P, P, P, P]),
    "gf_mask_rows": (I, [P, I, L, L, L, L, P, P]),
    "gf_mask_fill_sim": (I, [P, I, I, I, P, P, F, P]),
}


class GeoFormerLibError(RuntimeError):
    pass


_lib = None
_initialised_devices = set()


def load() -> ctypes.CDLL:
    """dlopen the library and bind every declared symbol (raises if the .so or a symbol is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GeoFormerLibError(
            f"{LIB_PATH} not found - build it with `python -m geoformer_b200.build` "
            "(there is no CPU or PyTorch fallback for the hot path)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.gf_abi_version() != 1:
        raise GeoFormerLibError("ABI version mismatch")
    _lib = lib
    return lib


def init(device_index: int) -> None:
    lib = load()
    if device_index in _initialised_devices:
        return
    rc = lib.gf_init(int(device_index))
    if rc != 0:
        raise GeoFormerLibError(f"gf_init({device_index}) failed: {lib.gf_last_error().decode()} (rc={rc})")
    _initialised_devices.add(device_index)


def call(name: str, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GeoFormerLibError(f"{name} failed: {lib.gf_last_error().decode()} (rc={rc})")


def launch_count() -> int:
    return int(load().gf_launch_count())
