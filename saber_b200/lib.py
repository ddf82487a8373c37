"""ctypes binding of ``libsaber_b200.so`` — the C ABI declared in ``include/saber_b200.h``.

There is no CPU fallback: if the library is missing it is built with nvcc; if that fails, or a
kernel call returns an error code, a ``RuntimeError`` carrying ``sb_last_error()`` is raised.
"""
from __future__ import annotations

import ctypes as C
import threading
from pathlib import Path

_LOCK = threading.Lock()
_LIB = None

c_void_p, c_int, c_ll, c_float, c_double = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_double

# name -> argtypes (every entry point returns int status unless listed in _SPECIAL)
SIGNATURES = {
    "sb_version": [],
    "sb_device_sm_count": [],
    "sb_require_sm100": [],
    "sb_gemm_bf16": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_void_p,
                     c_int, c_void_p, c_ll, c_int, c_int, c_float, c_int, c_void_p],
    "sb_gemm_set_prof": [c_void_p],
    "sb_gemm_ln": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_void_p, c_ll, c_int,
                   c_int, c_void_p, c_void_p, c_float, c_void_p],
    "sb_gemm_upscale1": [c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_void_p, c_ll, c_void_p,
                         c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_gemm_upscale2": [c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_void_p, c_ll, c_void_p,
                         c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_iou_gate": [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p],
    "sb_attention": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int,
                     c_int, c_int, c_int, c_float, c_int, c_int, c_void_p],
    "sb_attention_kadd": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int,
                          c_int, c_int, c_int, c_float, c_int, c_void_p],
    "sb_attention_few_keys": [c_void_p, c_ll, c_void_p, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int,
                              c_int, c_float, c_int, c_void_p],
    "sb_i2t_fold": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                    c_float, c_void_p],
    "sb_i2t_block_tc": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int,
                        c_int, c_int, c_void_p],
    "sb_t2i_tc_splits": [c_int, c_int],
    "sb_t2i_fold_attention_tc": [c_void_p, c_ll, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_float, c_void_p],
    "sb_mask_embed_keys": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "sb_window_attention": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_int, c_float, c_void_p],
    "sb_hiera_attention_tc": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p],
    "sb_hiera_attention_tc_prof": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p],
    "sb_layernorm": [c_void_p, c_ll, c_int, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_int, c_int,
                     c_float, c_int, c_void_p],
    "sb_im2col_k7s4": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "sb_im2col_k7s4_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "sb_gelu_exact_f32": [c_void_p, c_ll, c_void_p],
    "sb_rope_apply_f32": [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_attention_f32": [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int,
                         c_int, c_int, c_int, c_float, c_int, c_int, c_void_p],
    "sb_split3_bf16": [c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_ll, c_void_p],
    "sb_window_attention_f32": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                c_void_p],
    "sb_maxpool2x2": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "sb_add_upsample2x": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "sb_nhwc_to_nchw": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_nchw_to_nhwc": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "sb_add_cast": [c_void_p, c_int, c_void_p, c_ll, c_void_p, c_int, c_ll, c_void_p],
    "sb_prompt_tokens": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                         c_int, c_void_p, c_void_p],
    "sb_mask_downscale": [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_select_mask": [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p],
    "sb_amg_mask_post": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                         c_int, c_float, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                         c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_compact_keep": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sb_nms_dev": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p,
                   c_void_p, c_void_p],
    "sb_pair_intersections": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_void_p, c_void_p],
    "sb_unpack_bits": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_gather_rows": [c_void_p, c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "sb_amg_fill_lowres": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float, c_int, c_int, c_float,
                           c_float, c_void_p, c_void_p, c_int, c_void_p],
    "sb_amg_small_regions": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_int, c_void_p],
    "sb_masks_rle_size": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sb_masks_rle_counts": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_masks_rle_coco_size": [c_void_p, c_void_p, c_int, c_void_p, c_void_p],
    "sb_masks_rle_coco": [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    "sb_box_filter": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "sb_contrast_normalize": [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_float, c_void_p, c_void_p],
    "sb_rgb_mix_planar": [c_void_p, c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "sb_planar_to_hwc3": [c_void_p, c_ll, c_void_p, c_void_p],
    "sb_resize_normalize": [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, C.POINTER(c_float),
                            C.POINTER(c_float), c_void_p, c_void_p],
    "sb_upsample_bilinear": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_upsample_select": [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p],
    "sb_resample_frames_u8": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                              c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_stitch_labels": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_ccl3d_26": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_ccl3d": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_rope_apply": [c_void_p, c_ll, c_int, c_void_p, c_ll, c_ll, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_conv3x3s2_ln_gelu": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                             c_int, c_float, c_float, c_void_p, c_void_p],
    "sb_im2col_3x3s2": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_dwconv7_ln": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p,
                      c_void_p],
    "sb_add_vec_cond": [c_void_p, c_void_p, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p],
    "sb_track_select": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                        c_void_p, c_void_p, c_void_p],
    "sb_objptr_mix": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    "sb_fill_holes": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_threshold_affine": [c_void_p, c_float, c_float, c_float, c_ll, c_void_p, c_void_p],
    "sb_conv4x4s4": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_stitch_objects": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_slice_any": [c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "sb_erase_label": [c_void_p, c_ll, c_int, c_void_p],
    "sb_minmax": [c_void_p, c_ll, c_void_p, c_void_p, c_void_p],
    "sb_minmax_affine": [c_void_p, c_ll, c_void_p, c_float, c_float, c_float, c_void_p, c_void_p],
    "sb_zoom_linear_mirror": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p],
    "sb_gauss1d_mirror": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p],
    "sb_gaussian_z": [c_void_p, c_int, c_ll, c_void_p, c_int, c_void_p, c_void_p],
    "sb_mean_z": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p],
    "sb_mean_std": [c_void_p, c_ll, c_void_p, c_void_p, c_void_p],
    "sb_standardize": [c_void_p, c_ll, c_void_p, c_void_p, c_void_p],
    "sb_mask_bbox": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_crop_resize": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "sb_mask_features": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_prelu": [c_void_p, c_int, c_ll, c_float, c_void_p, c_void_p],
    "sb_im2col_3x3s1": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_mean_tokens": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_softmax_rows": [c_void_p, c_int, c_int, c_void_p, c_void_p],
    "sb_label_equals": [c_void_p, c_int, c_ll, C.c_uint, c_void_p, c_void_p, c_void_p],
    "sb_corr1d_zero": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p],
    "sb_threshold_label": [c_void_p, c_ll, c_float, c_int, c_void_p, c_void_p],
    "sb_morph_ball": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_morph_cube": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_fft_twiddles": [c_int, c_void_p, c_void_p],
    "sb_fft_lines": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_ll, c_int, c_int, c_int, c_int, c_float, c_int, c_int,
                     c_void_p, c_int, c_int, c_int, c_void_p],
    "sb_bandpass_volume": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "sb_trim_binarize": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "sb_z_any": [c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "sb_label_bbox": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p],
    "sb_roi_binarize": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_ll, c_void_p,
                        c_void_p, c_void_p],
    "sb_roi_paste": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_ll,
                     c_void_p],
    "sb_overlay_nonzero": [c_void_p, c_void_p, c_int, c_ll, c_void_p],
    "sb_mask_logic": [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p],
    "sb_label_select": [c_void_p, c_ll, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    "sb_label_keep_ratio": [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p],
}


def lib_path() -> Path:
    return Path(__file__).resolve().parent / "libsaber_b200.so"


def load() -> C.CDLL:
    """Load (building first if needed) the CUDA library. Raises if it cannot be produced."""
    global _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        path = lib_path()
        from . import build as _build
        # always consult the source digest: build() returns at once when the library matches csrc/ (a stale library
        # after a pull would silently keep the old kernels); a box without nvcc uses the shipped library as is
        try:
            _build.build()
        except RuntimeError:
            if not path.exists():
                raise
        lib = C.CDLL(str(path))
        lib.sb_last_error.restype = C.c_char_p
        lib.sb_last_error.argtypes = []
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError => missing symbol: fail loudly
            fn.argtypes = argtypes
            fn.restype = c_int
        _LIB = lib
        return lib


def last_error() -> str:
    return load().sb_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc < 0:
        raise RuntimeError(f"saber_b200 {what} failed (code {rc}): {last_error()}")
