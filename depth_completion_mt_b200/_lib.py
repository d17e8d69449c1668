"""ctypes binding of the C ABI declared in include/dcmt.h.

``load()`` opens depth_completion_mt_b200/libdcmt.so (built by ``depth_completion_mt_b200.build``).
There is deliberately no fallback: if the CUDA library is missing or does not load, importing the
compute API raises.  ``bind(path)`` is what ``load`` uses internally; the test-suite also uses it to
bind the CPU emulator build of the same sources (tests/emu) -- the product never does.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libdcmt.so")

DCMT_OK, DCMT_E_BADARG, DCMT_E_UNSUPPORTED, DCMT_E_CUDA, DCMT_E_NOMEM = 0, -1, -2, -3, -4
BLUR = {"none": 0, "gaussian": 1, "bilateral": 2}
PATH = {"auto": 0, "generic": 1, "fused": 2, "rank": 3}
STATS_STRIDE = 4
N_STAGES = 10


class StereoParams(C.Structure):
    """dcmt_stereo_params (include/dcmt.h); defaults = main_sl.cpp literals."""

    _fields_ = [
        ("baseline", C.c_float), ("focal", C.c_float), ("damp_factor", C.c_float), ("err_clip", C.c_float),
        ("depth_clip", C.c_float), ("num_iterations", C.c_int32), ("final_gauss", C.c_int32),
    ]


class EvalResult(C.Structure):
    """dcmt_eval_result (include/dcmt.h)."""

    _fields_ = [("count", C.c_double), ("sum_err", C.c_double), ("sum_abs", C.c_double), ("sum_sq", C.c_double),
                ("mean_err", C.c_float), ("mae", C.c_float), ("rmse", C.c_float), ("pad", C.c_int32)]


class KittiMetrics(C.Structure):
    """dcmt_kitti_metrics (include/dcmt.h)."""

    _fields_ = [("n_gt", C.c_double), ("n_pred", C.c_double), ("n_unfilled", C.c_double), ("sum_abs", C.c_double),
                ("sum_sq", C.c_double), ("sum_iabs", C.c_double), ("sum_isq", C.c_double), ("mae_mm", C.c_float),
                ("rmse_mm", C.c_float), ("imae_per_km", C.c_float), ("irmse_per_km", C.c_float), ("density", C.c_float),
                ("pad", C.c_int32)]


class DcmtError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"dcmt status {status}: {message}")
        self.status = status


_P = C.c_void_p
_SIGNATURES = {
    "dcmt_version": (C.c_int, []),
    "dcmt_build_info": (C.c_char_p, []),
    "dcmt_last_error": (C.c_char_p, []),
    "dcmt_status_string": (C.c_char_p, [C.c_int]),
    "dcmt_device_count": (C.c_int, []),
    "dcmt_release_workspaces": (C.c_int, []),
    "dcmt_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dcmt_launch_count": (C.c_longlong, []),
    "dcmt_host_alloc": (C.c_int, [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "dcmt_host_free": (C.c_int, [_P]),
    "dcmt_profile_begin": (C.c_int, []),
    "dcmt_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "dcmt_img_completion_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_img_completion_f32_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_img_completion_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_img_completion_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_interpolate_with_superpixels_f32": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, _P, _P]),
    "dcmt_interpolate_with_superpixels_f32_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, _P]),
    "dcmt_interpolate_with_superpixels_ex_f32": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_interpolate_with_superpixels_ex_f32_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_stereo_params_default": (None, [C.POINTER(StereoParams)]),
    "dcmt_stereo_params_official": (None, [C.POINTER(StereoParams), C.c_int]),
    "dcmt_stereo_refine_f32": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(StereoParams), _P]),
    "dcmt_stereo_refine_f32_host": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(StereoParams)]),
    "dcmt_measurement_derivatives_f32": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_get_initial_disparity_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, _P]),
    "dcmt_optimize_ig_f32": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, _P]),
    "dcmt_retrieve_optimized_depth_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, _P]),
    "dcmt_evaluate_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P, _P]),
    "dcmt_evaluate_f32_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P]),
    "dcmt_evaluate_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P, _P]),
    "dcmt_evaluate_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P]),
    "dcmt_evaluate_u16_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P, _P]),
    "dcmt_evaluate_u16_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, _P]),
    "dcmt_evaluate_kitti_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P, _P]),
    "dcmt_evaluate_kitti_f32_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_evaluate_kitti_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P, _P]),
    "dcmt_evaluate_kitti_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_evaluate_kitti_u16_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P, _P]),
    "dcmt_evaluate_kitti_u16_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_lidar_project_f32": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, C.c_float, C.c_float, _P, _P]),
    "dcmt_lidar_project_batch_f32": (C.c_int, [_P, _P, C.c_int, C.c_size_t, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, C.c_float, C.c_float, _P, _P]),
    "dcmt_lidar_project_f32_host": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, C.c_float, C.c_float, _P]),
    "dcmt_slic_center_count": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dcmt_slic_u8c3": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "dcmt_slic_u8c3_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_slic_bgr_u8c3": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "dcmt_slic_bgr_u8c3_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_img_completion_f32_host_multi": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_img_completion_u16_host_multi": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_interpolate_with_superpixels_f32_host_multi": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_debug_host_copy_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "dcmt_debug_host_copy_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "dcmt_debug_host_copy_u16_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "dcmt_img_completion_u16_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_img_completion_u16_u16_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_img_completion_u16_u16_host_multi": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_interpolate_with_superpixels_u16": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_interpolate_with_superpixels_u16_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_interpolate_with_superpixels_u16_host_multi": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_interpolate_with_superpixels_u16_u16": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P]),
    "dcmt_interpolate_with_superpixels_u16_u16_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P]),
    "dcmt_interpolate_with_superpixels_u16_u16_host_multi": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "dcmt_depth_to_u16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_bgr2gray_u8": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_bgr2gray_u8_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int]),
    "dcmt_bgr2lab_u8": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "dcmt_bgr2lab_u8_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int]),
    "dcmt_entries_measurement_derivatives": (C.c_int, [_P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, _P]),
    "dcmt_entries_measurement_derivatives_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_size_t, C.c_size_t]),
    "dcmt_entries_optimize_ig": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, _P]),
    "dcmt_entries_optimize_ig_host": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float]),
    "dcmt_get_initial_disparity_mat_f32": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_float, C.c_float, _P]),
    "dcmt_get_initial_disparity_mat_f32_host": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_float, C.c_float]),
    "dcmt_retrieve_optimized_depth_mat_f32": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, _P]),
    "dcmt_retrieve_optimized_depth_mat_f32_host": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]),
    "dcmt_debug_q8_phase_cycles": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, C.POINTER(C.c_int), _P]),
    "dcmt_img_completion_stages_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.POINTER(C.c_uint32), _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class Library:
    """A loaded libdcmt with typed entry points; ``check`` turns status codes into DcmtError."""

    def __init__(self, path: str):
        self.path = path
        self.cdll = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(self.cdll, name)  # AttributeError = symbol missing: fail loudly
            fn.restype = res
            fn.argtypes = args
            setattr(self, name, fn)

    def check(self, status: int) -> None:
        if status != DCMT_OK:
            raise DcmtError(status, self.dcmt_last_error().decode("utf-8", "replace"))


def bind(path: str) -> Library:
    return Library(path)


_default: Library | None = None


def _product(path: str) -> Library:
    lib = Library(path)
    info = lib.dcmt_build_info().decode()
    if not info.startswith("cuda"):  # e.g. the CPU emulator build of tests/emu: test infrastructure, never the product
        raise ImportError(f"{path} is not a CUDA build of libdcmt ({info!r}); depth_completion_mt_b200 has no CPU fallback.")
    return lib


def load() -> Library:
    """The product library.  Raises if libdcmt.so is absent -- there is no CPU fallback.  ``load().path`` names the file
    that was bound (bench.py prints it)."""
    global _default
    if _default is None:
        alt = os.environ.get("DCMT_LIB")  # A/B builds of the same sources (tools/build_variant.py); must be a CUDA build
        if alt:
            _default = _product(alt)
            return _default
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m depth_completion_mt_b200.build` "
                "(nvcc, sm_100a). depth_completion_mt_b200 has no CPU fallback.")
        _default = _product(LIB_PATH)
    return _default
