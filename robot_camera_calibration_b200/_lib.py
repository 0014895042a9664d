"""ctypes binding of the C ABI declared in include/rcc_ba.h.

There is no fallback: if librcc_ba.so is missing (or cannot be loaded) every
use of the package fails loudly with the build instruction.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RCC_BA_LIB") or os.path.join(HERE, "librcc_ba.so")   # override: kernel-variant experiments

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)
c_int16_p = C.POINTER(C.c_int16)

RCC_OK, RCC_BAD_ARG, RCC_CUDA_ERROR, RCC_NCCL_ERROR, RCC_EVAL_FAILED, RCC_NOT_SPD, RCC_NOT_READY, RCC_SOLVER_ERROR = range(8)
STATUS_NAMES = ["RCC_OK", "RCC_BAD_ARG", "RCC_CUDA_ERROR", "RCC_NCCL_ERROR", "RCC_EVAL_FAILED", "RCC_NOT_SPD",
                "RCC_NOT_READY", "RCC_SOLVER_ERROR"]
MODEL_SINGLE, MODEL_RIG = 0, 1
ELIM_AUTO, ELIM_VIEWS, ELIM_MARKERS = 0, 1, 2
BLOCK_VIEW, BLOCK_MARKER, BLOCK_INTR, BLOCK_DIST, BLOCK_EXT = range(5)
LENS_RADTAN, LENS_EQUIDISTANT = 0, 1
LENSES = {"radtan": LENS_RADTAN, "equidistant": LENS_EQUIDISTANT}
COMM_ID_BYTES = 128


class Options(C.Structure):
    _fields_ = [("model", C.c_int32), ("n_views", C.c_int32), ("n_markers", C.c_int32),
                ("n_cameras", C.c_int32), ("n_obs_blocks", C.c_int64), ("device", C.c_int32),
                ("eliminate", C.c_int32)]


class LMOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("initial_radius", C.c_double), ("max_radius", C.c_double),
                ("min_relative_decrease", C.c_double), ("function_tolerance", C.c_double),
                ("gradient_tolerance", C.c_double), ("parameter_tolerance", C.c_double),
                ("min_diagonal", C.c_double), ("max_diagonal", C.c_double), ("verbose", C.c_int32),
                ("jacobi_scaling", C.c_int32)]


class LMSummary(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("accepted", C.c_int32), ("termination", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double), ("final_gradient_max", C.c_double),
                ("final_radius", C.c_double), ("total_ms", C.c_double), ("linearize_ms", C.c_double),
                ("schur_ms", C.c_double), ("allreduce_ms", C.c_double), ("solve_ms", C.c_double),
                ("backsub_ms", C.c_double), ("cost_ms", C.c_double)]


class Dims(C.Structure):
    _fields_ = [("eliminated_is_view", C.c_int32), ("n_e", C.c_int32), ("n_f", C.c_int32),
                ("n_shared", C.c_int32), ("n_reduced", C.c_int32), ("ld_reduced", C.c_int32),
                ("n_pairs", C.c_int64)]


# every symbol include/rcc_ba.h declares: name -> (restype, argtypes)
_H = C.c_void_p
SIGNATURES = {
    "rcc_ba_create": (C.c_int, [C.POINTER(Options), C.POINTER(_H)]),
    "rcc_ba_destroy": (None, [_H]),
    "rcc_ba_last_error": (C.c_char_p, [_H]),
    "rcc_lm_default_options": (None, [C.POINTER(LMOptions)]),
    "rcc_ba_version": (C.c_char_p, []),
    "rcc_ba_set_stream": (C.c_int, [_H, C.c_void_p]),
    "rcc_ba_set_intrinsics": (C.c_int, [_H, c_double_p, c_double_p]),
    "rcc_ba_set_rig_extrinsics": (C.c_int, [_H, c_double_p]),
    "rcc_ba_set_view_poses": (C.c_int, [_H, c_double_p]),
    "rcc_ba_set_marker_poses": (C.c_int, [_H, c_double_p]),
    "rcc_ba_set_marker_sizes": (C.c_int, [_H, c_double_p]),
    "rcc_ba_set_observations": (C.c_int, [_H, c_int32_p, c_int32_p, c_int32_p, c_double_p]),
    "rcc_ba_update_pixels": (C.c_int, [_H, c_double_p]),
    "rcc_ba_set_observations_i16": (C.c_int, [_H, c_int32_p, c_int32_p, c_int32_p, c_int16_p]),
    "rcc_ba_set_observations_i32": (C.c_int, [_H, c_int32_p, c_int32_p, c_int32_p, c_int32_p]),
    "rcc_ba_update_pixels_i16": (C.c_int, [_H, c_int16_p]),
    "rcc_ba_set_constant": (C.c_int, [_H, C.c_int32, C.c_int32, C.c_int32]),
    "rcc_ba_set_loss": (C.c_int, [_H, C.c_int32, C.c_double]),
    "rcc_ba_set_lens": (C.c_int, [_H, C.c_int32]),
    "rcc_ba_set_camera_lenses": (C.c_int, [_H, c_int32_p]),
    "rcc_ba_set_corner_layout": (C.c_int, [_H, C.c_int32, c_double_p, c_int32_p]),
    "rcc_ba_set_priors": (C.c_int, [_H, C.c_int32, C.c_int64, c_int32_p, c_double_p, c_double_p]),
    "rcc_ba_get_intrinsics": (C.c_int, [_H, c_double_p, c_double_p]),
    "rcc_ba_get_rig_extrinsics": (C.c_int, [_H, c_double_p]),
    "rcc_ba_get_view_poses": (C.c_int, [_H, c_double_p]),
    "rcc_ba_get_marker_poses": (C.c_int, [_H, c_double_p]),
    "rcc_ba_evaluate": (C.c_int, [_H, C.c_int32, c_double_p] + [c_double_p] * 6),
    "rcc_ba_evaluate_device": (C.c_int, [_H, C.c_int32, c_double_p]),
    "rcc_ba_linearize": (C.c_int, [_H, c_double_p]),
    "rcc_ba_schur": (C.c_int, [_H, C.c_double]),
    "rcc_ba_set_lm_diagonal": (C.c_int, [_H, C.c_double, C.c_double, C.c_int32]),
    "rcc_ba_solve_step": (C.c_int, [_H, c_double_p, c_double_p, c_double_p]),
    "rcc_ba_candidate_cost": (C.c_int, [_H, c_double_p]),
    "rcc_ba_accept_step": (C.c_int, [_H]),
    "rcc_ba_solve": (C.c_int, [_H, C.POINTER(LMOptions), C.POINTER(LMSummary)]),
    "rcc_ba_covariance": (C.c_int, [_H, c_double_p, c_double_p, c_double_p]),
    "rcc_ba_covariance_blocks": (C.c_int, [_H, C.c_int64, c_int32_p, c_double_p]),
    "rcc_ba_get_dims": (C.c_int, [_H, C.POINTER(Dims)]),
    "rcc_ba_get_normal_blocks": (C.c_int, [_H] + [c_double_p] * 9),
    "rcc_ba_get_reduced_system": (C.c_int, [_H, c_double_p, c_double_p]),
    "rcc_ba_get_reduced_block": (C.c_int, [_H, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_double_p]),
    "rcc_ba_get_step": (C.c_int, [_H, c_double_p, c_double_p, c_double_p]),
    "rcc_comm_get_unique_id": (C.c_int, [C.c_char_p]),
    "rcc_ba_comm_init": (C.c_int, [_H, C.c_char_p, C.c_int32, C.c_int32]),
    "rcc_ba_profile_enable": (C.c_int, [_H, C.c_int32]),
    "rcc_ba_profile_reset": (C.c_int, [_H]),
    "rcc_ba_profile_get": (C.c_int, [_H, C.c_char_p, c_double_p, c_int64_p]),
    "rcc_ba_launch_count": (C.c_int64, [_H]),
    "rcc_ba_synchronize": (C.c_int, [_H]),
    "rcc_ba_flush_l2": (C.c_int, [_H]),
    "rcc_dense_potrf": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_int32_p,
                                  c_double_p]),
    "rcc_dense_trsv": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, c_double_p]),
    "rcc_fp64_peak_tflops": (C.c_int, [C.c_int32, c_double_p]),
    "rcc_pnp_batch": (C.c_int, [C.c_int32, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                C.c_int32]),
    "rcc_pnp_batch_lens": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p,
                                     c_double_p, C.c_int32]),
    "rcc_pnp_target_batch": (C.c_int, [C.c_int32, C.c_int32, c_double_p, C.c_int32, c_double_p, C.c_int64, c_int64_p,
                                       c_int32_p, c_double_p, c_double_p, c_double_p, C.c_int32]),
    "rcc_homography_target_batch": (C.c_int, [C.c_int32, C.c_int32, c_double_p, C.c_int64, c_int64_p, c_int32_p,
                                              c_double_p, c_double_p, c_double_p, C.c_int32]),
}

_lib = None


class RccError(RuntimeError):
    def __init__(self, status, message):
        name = STATUS_NAMES[status] if 0 <= status < len(STATUS_NAMES) else str(status)
        super().__init__(f"{name}: {message}")
        self.status = status


def load():
    """Load librcc_ba.so and bind every declared entry point.  Raises if the
    library has not been built -- there is deliberately no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m robot_camera_calibration_b200._build` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
