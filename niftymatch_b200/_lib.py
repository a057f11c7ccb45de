"""ctypes binding of the C-ABI (include/nm_b200.h) in niftymatch_b200/libnm_b200.so.

The product path has no CPU fallback: if the shared library is missing or a compute call
fails, an exception is raised.  Nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnm_b200.so")


class NmError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"{what}: nm error {code}: {strerror(code)}")
        self.code = code


class SiftParamsC(C.Structure):
    """struct nm_sift_params (mirror of the reference's class SiftParams)."""
    _fields_ = [
        ("width", C.c_int), ("height", C.c_int),
        ("num_octaves", C.c_int), ("num_dog_levels", C.c_int),
        ("level_max", C.c_int), ("level_min", C.c_int),
        ("sigma_d_0", C.c_float), ("sigma_k", C.c_float), ("sigma_0", C.c_float), ("sigma_n", C.c_float),
        ("base_smooth", C.c_float),
        ("sigmas", C.c_float * 8),
        ("num_sigmas", C.c_int),
        ("peak_threshold", C.c_float), ("edge_threshold", C.c_float),
    ]


_vp, _i, _f, _ull = C.c_void_p, C.c_int, C.c_float, C.c_ulonglong

# name -> (restype, argtypes).  Every symbol include/nm_b200.h declares is listed here;
# tests/test_abi.py checks header <-> table <-> shared library agree.
SIGNATURES = {
    "nm_strerror": (C.c_char_p, [_i]),
    "nm_device_cc": (_i, []),
    "nm_version": (C.c_char_p, []),
    "nm_selftest_gradient": (_i, [C.c_longlong, C.c_uint, C.POINTER(C.c_longlong)]),
    "nm_sift_params_init": (_i, [C.POINTER(SiftParamsC), _i, _i]),
    "nm_gaussian_taps": (_i, [_f, _vp, C.POINTER(_i)]),
    "nm_blur_f32": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _vp]),
    "nm_downsample2_f32": (_i, [_vp, _i, _i, _vp, _i, _i, _vp]),
    "nm_subtract_f32": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "nm_gradient_f32": (_i, [_vp, _vp, _i, _i, _vp]),
    "nm_keypoints_dense_f32": (_i, [_vp, _vp, _vp, _i, _i, _f, _f, _f, _f, _i, _i, _vp, _vp]),
    "nm_keypoints_dense_masked_f32": (_i, [_vp, _vp, _vp, _ull, _i, _i, _f, _f, _f, _f, _i, _i, _vp, _vp]),
    "nm_keypoints_dense_tex": (_i, [_ull, _ull, _ull, _ull, _i, _i, _f, _f, _f, _f, _i, _i, _vp, _vp]),
    "nm_collate_f32": (_i, [_vp, _i, _vp, _vp, _vp]),
    "nm_orientations_f32": (_i, [_vp, _vp, _i, _i, _i, _f, _f, _vp, _vp]),
    "nm_descriptors_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp]),
    "nm_transpose_f32": (_i, [_vp, _vp, _i, _i, _vp]),
    "nm_dist2_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp]),
    "nm_set_matches_f32": (_i, [_vp, _i, _i, _i, _vp, _f, _vp]),
    "nm_match_f32": (_i, [_vp, _i, _vp, _i, _f, _vp, _vp, _vp]),
    "nm_match_top2_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp]),
    "nm_match_merge_top2": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "nm_match_merge_top2_strided": (_i, [_vp, _i, C.c_longlong, _i, _f, _vp, _vp]),
    "nm_match_pairs_f32": (_i, [_vp, _vp, _i, _i, _f, _vp, _vp, _vp, _vp]),
    "nm_match_pairs_span_f32": (_i, [_vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp, _vp]),
    "nm_match_tc_probe": (_i, [_vp, _i, _vp, _i, _vp, C.POINTER(_i), _vp, _vp, C.POINTER(_i), C.POINTER(_f), _vp]),
    "nm_grayscale_bgra_f32": (_i, [_vp, _vp, _i, _i, _vp]),
    "nm_bgra_extract_channel_f32": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "nm_bgra_put_channel_f32": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "nm_bgra_set_alpha": (_i, [_vp, _i, _i, C.c_ubyte, _vp]),
    "nm_cast_f32_u8": (_i, [_vp, _i, _i, _vp, C.c_ubyte, _vp]),
    "nm_undistort_map_f32": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_resample_tex_f32": (_i, [_ull, _vp, _vp, _i, _i, _vp, _vp]),
    "nm_resample_perspective_bgra": (_i, [_vp, _ull, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "nm_resample_mask_tex_u8": (_i, [_vp, _ull, _i, _i, _vp, _vp, _f, _vp]),
    "nm_transform_blend_bgra": (_i, [_vp, _i, _i, _ull, _i, _i, _i, _i, _vp, _i, _i, _ull, _vp, _ull, _vp]),
    "nm_mosaic_create": (_i, [C.POINTER(_vp), _i, _i, _i, _vp, _vp]),
    "nm_mosaic_destroy": (_i, [_vp]),
    "nm_mosaic_place_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_mosaic_blend_bgra": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "nm_mosaic_textures": (_i, [_vp, C.POINTER(_ull), C.POINTER(_ull), C.POINTER(_ull)]),
    "nm_sift_run_bgra": (_i, [_vp, _vp, _i, _vp]),
    "nm_align_points_f32": (_i, [_vp] * 9 + [_i, _vp]),
    "nm_align_pairs_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_align_pairs_span_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_ransac_hypotheses_f32": (_i, [_i, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp, _vp, _vp]),
    "nm_ransac_f32": (_i, [_i, _vp, _vp, _vp, _vp, _i, _f, _i, _ull, _vp, _vp, _vp]),
    "nm_ransac_batch_f32": (_i, [_i, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _i, _i, _f, _i, _ull, _vp, _vp, _vp]),
    "nm_ransac_refine_batch_f32": (_i, [_i, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _i, _i, _f, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "nm_ransac_adjust_chain_f32": (_i, [_i, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp, _i,
                                        _vp, _vp, _vp, _vp, _vp]),
    "nm_ransac_adjust_chain_cost_f32": (_i, [_i, _i, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp,
                                             _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_ransac_adjust_chain_fixed_f32": (_i, [_i, _i, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp,
                                              _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_match_set_engine": (_i, [_i]),
    "nm_match_get_engine": (_i, []),
    "nm_sift_create": (_i, [C.POINTER(_vp), C.POINTER(SiftParamsC), _i, _i]),
    "nm_sift_destroy": (_i, [_vp]),
    "nm_sift_run": (_i, [_vp, _vp, _i, _vp]),
    "nm_sift_set_mask": (_i, [_vp, _ull]),
    "nm_sift_set_mask_image": (_i, [_vp, _vp, _i, _i]),
    "nm_sift_run_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_sift_results": (_i, [_vp] + [C.POINTER(_vp)] * 7),
    "nm_sift_level": (_i, [_vp, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "nm_sift_grad": (_i, [_vp, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "nm_sift_last_launches": (_i, [_vp]),
    "nm_sift_enable_timing": (_i, [_vp, _i]),
    "nm_sift_stage_ms": (_i, [_vp, _vp]),
    "nm_sift_stage_ms7": (_i, [_vp, _vp]),
    "nm_sift_set_dense_gradients": (_i, [_vp, _i]),
    "nm_sift_set_exact_descriptor": (_i, [_vp, _i]),
}

_lib = None


def load() -> C.CDLL:
    """Load libnm_b200.so (built in-tree by `make` / __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first (`make` or "
                "`python -c 'import __graft_entry__ as g; g.build()'`).  There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def strerror(code: int) -> str:
    try:
        return load().nm_strerror(code).decode()
    except Exception:  # pragma: no cover
        return "?"


def check(code: int, what: str) -> None:
    if code != 0:
        raise NmError(code, what)
