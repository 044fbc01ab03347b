"""ctypes binding of the C-ABI library ``csrc/libnirgan_b200.so`` (see ``include/nirgan_b200.h``).

There is no CPU fallback: if the shared library is missing, or a call returns a non-zero status, a
``RuntimeError`` carrying ``ng_last_error()`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libnirgan_b200.so")

# enums of include/nirgan_b200.h
F32, F16, BF16, U16 = 0, 1, 2, 3
IMPL_SIMT, IMPL_TC = 0, 1
FORM_GATHER, FORM_PHASED, FORM_PHASED_MERGED = 0, 1, 2
EPI_RAW, EPI_BIAS_ACT, EPI_HEAD = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH = 0, 1, 2, 3
HALO_ZERO, HALO_REFLECT = 0, 1
INJECT_NONE, INJECT_ADD, INJECT_MUL_SCALED, INJECT_MUL = 0, 1, 2, 3

c_i32, c_i64, c_f32, c_vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p
ABI_VERSION = 102          # NG_VERSION of include/nirgan_b200.h this binding was written against


class ConvArgs(C.Structure):
    """Mirror of ``struct ng_conv_args``."""
    _fields_ = [(n, c_i32) for n in (
        "dtype", "impl", "form", "sgn", "B", "Hin", "Win", "Cin", "in_pad", "in_pad_w", "Cout", "KH", "KW", "stride",
        "pad", "pad_w", "Hout", "Wout", "epilogue", "act")] + [
        ("slope", c_f32), ("crop", c_i32), ("reserved", c_i32),
        ("x", c_vp), ("w", c_vp), ("bias", c_vp), ("y", c_vp), ("stat_partials", c_vp),
        ("mean_rstd", c_vp), ("tile_counters", c_vp), ("stat_acc", c_vp)]


_SIGNATURES = {
    "ng_version": (c_i32, []),
    "ng_last_error": (C.c_char_p, []),
    "ng_device_check": (c_i32, [c_i32]),
    "ng_conv_stat_slots": (c_i32, [C.POINTER(ConvArgs)]),
    "ng_conv2d": (c_i32, [C.POINTER(ConvArgs), c_vp]),
    "ng_conv2d_wgrad_workspace_bytes": (c_i64, [C.POINTER(ConvArgs)]),
    "ng_conv2d_wgrad": (c_i32, [C.POINTER(ConvArgs), c_vp, c_vp, c_vp, c_i64, c_vp]),
    "ng_pack_weight": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_unpack_weight_grad": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_f32, c_vp,
                                      c_vp]),
    "ng_pack_weight_phasemerged": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_prep_stem": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_pack_weight_rowmerged": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_stem_conv": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "ng_stem_conv_stat_slots": (c_i32, [c_i32, c_i32, c_i32]),
    "ng_unpack_weight_grad_rowmerged": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_f32, c_vp, c_vp]),
    "ng_head_conv": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "ng_tap_gather": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "ng_tap_scatter": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_i32, c_vp,
                               c_vp]),
    "ng_prep_input": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32,
                              c_vp, c_vp]),
    "ng_in_stats": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_in_stats_finalize": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_in_apply": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_f32, c_vp, c_i32, c_vp,
                            c_i32, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "ng_memset_zero": (c_i32, [c_vp, c_i64, c_vp]),
    "ng_in_bwd_scratch_floats": (c_i64, [c_i32, c_i32, c_i32, c_i32]),
    "ng_in_bwd": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_f32, c_vp,
                          c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "ng_grad_scale_pow2": (c_i32, [c_vp, c_i64, c_f32, c_vp, c_vp]),
    "ng_head_bwd_prep": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "ng_grad_to_nchw": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp]),
    "ng_prep_input_s2d": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_pack_weight_s2d": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_unpack_weight_grad_s2d": (c_i32, [c_vp, c_i32, c_i32, c_f32, c_vp, c_f32, c_vp, c_vp]),
    "ng_inject_bwd": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "ng_resize_plane": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_hist_match_workspace_bytes": (c_i64, [c_i32, c_i32, c_i32]),
    "ng_hist_match": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_i64, c_vp]),
    "ng_sort_segments": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp, c_i64, c_vp]),
    "ng_image_metrics_scratch_floats": (c_i64, [c_i32, c_i32, c_i32]),
    "ng_image_metrics": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp]),
    "ng_ssim_loss_scratch_floats": (c_i64, [c_i32, c_i32, c_i32]),
    "ng_ssim_loss": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "ng_emd_loss": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "ng_scene_tiles": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_f32, c_vp, c_vp]),
    "ng_scene_blend": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_scene_tile_valid": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_f32, c_vp, c_vp]),
    "ng_scene_blend_masked": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32,
                                      c_i32, c_i32, c_i32, c_f32, c_f32, c_vp, c_vp]),
    "ng_scene_blend_indices": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp,
                                       c_i32, c_i32, c_i32, c_i32, c_f32, c_i32, c_f32, c_f32, c_vp, c_i32, c_vp, c_vp]),
    "ng_satclip_encode": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_i32, c_i32, c_i32, C.c_double, C.c_double, c_vp, c_vp]),
    "ng_linear": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "ng_lsgan_loss": (c_i32, [c_vp, c_i64, c_f32, c_vp, c_i32, c_vp, c_f32, c_vp]),
    "ng_rs_pixel_losses": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "ng_rs_index": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "ng_adam_multi": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_vp, c_f32,
                              c_vp, c_vp]),
    "ng_nonfinite_flag": (c_i32, [c_vp, c_i64, c_vp, c_vp]),
    "ng_adam_step": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_i32, c_f32, c_vp]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load (once) and return the ctypes library.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"nirgan_b200: native library {LIB_PATH} not found. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (or nir-gan_b200/csrc/build.sh). "
            f"There is no CPU / PyTorch fallback for the hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    got = lib.ng_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"nirgan_b200: {LIB_PATH} reports C-ABI version {got}, this binding needs {ABI_VERSION}: "
                           f"rebuild it (nir-gan_b200/csrc/build.sh)")
    _lib = lib
    return lib


def last_error() -> str:
    return load().ng_last_error().decode("utf-8", "replace")


def check(status: int, what: str = "") -> None:
    if status != 0:
        raise RuntimeError(f"nirgan_b200 {what} failed with status {status}: {last_error()}")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
