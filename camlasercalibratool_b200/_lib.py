"""ctypes declarations for the C ABI of libclc_b200.so (include/clc_b200.h).

Loading fails loudly: there is no CPU or pure-Python fallback for any entry point.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)


class ClcError(RuntimeError):
    pass


class ProblemDesc(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int64),
        ("frame_pose", c_double_p),
        ("offsets", c_int64_p),
        ("points", c_double_p),
        ("edge_points", c_double_p),
        ("use_loss", C.c_int),
        ("cauchy_a", C.c_double),
        ("device", C.c_int),
    ]


class GatherDesc(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int64),
        ("frame_pose", c_double_p),
        ("frame_points", C.POINTER(c_double_p)),
        ("frame_counts", c_int64_p),
        ("edge_points", c_double_p),
        ("use_loss", C.c_int),
        ("cauchy_a", C.c_double),
        ("device", C.c_int),
    ]


class SyntheticDesc(C.Structure):
    _fields_ = [
        ("n_frames_total", C.c_int64),
        ("frame_begin", C.c_int64),
        ("frame_end", C.c_int64),
        ("beams", C.c_int64),
        ("seed", C.c_uint64),
        ("sigma", C.c_double),
        ("with_edges", C.c_int),
        ("use_loss", C.c_int),
        ("cauchy_a", C.c_double),
        ("device", C.c_int),
        ("camera_model", C.c_int),
        ("camera_intrinsics", C.c_double * 8),
        ("pixel_sigma", C.c_double),
        ("image_width", C.c_int),
        ("image_height", C.c_int),
        ("grid_rows", C.c_int),
        ("grid_cols", C.c_int),
        ("tag_size", C.c_double),
        ("tag_spacing", C.c_double),
    ]


class CameraDesc(C.Structure):
    _fields_ = [
        ("camera_model", C.c_int),
        ("intrinsics", C.c_double * 8),
        ("grid_rows", C.c_int),
        ("grid_cols", C.c_int),
        ("tag_size", C.c_double),
        ("tag_spacing", C.c_double),
    ]


class ScanDesc(C.Structure):
    _fields_ = [
        ("n_scans", C.c_int64),
        ("n_beams", C.c_int64),
        ("ranges", C.POINTER(C.c_float)),
        ("scan_stamp", c_double_p),
        ("angle_min", C.c_double),
        ("angle_increment", C.c_double),
        ("range_min", C.c_double),
        ("n_poses", C.c_int64),
        ("pose_stamp", c_double_p),
        ("pose_wc", c_double_p),
        ("max_dt", C.c_double),
        ("line_fit_max_iterations", C.c_int),
        ("with_edges", C.c_int),
        ("use_loss", C.c_int),
        ("cauchy_a", C.c_double),
        ("device", C.c_int),
    ]


class LmOptions(C.Structure):
    _fields_ = [
        ("max_num_iterations", C.c_int),
        ("initial_trust_region_radius", C.c_double),
        ("max_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double),
        ("min_relative_decrease", C.c_double),
        ("min_lm_diagonal", C.c_double),
        ("max_lm_diagonal", C.c_double),
        ("function_tolerance", C.c_double),
        ("gradient_tolerance", C.c_double),
        ("parameter_tolerance", C.c_double),
        ("max_num_consecutive_invalid_steps", C.c_int),
        ("jacobi_scaling", C.c_int),
        ("iterations_per_sync", C.c_int),
        ("reserved", C.c_int),
    ]


class LmIteration(C.Structure):
    _fields_ = [
        ("iteration", C.c_int),
        ("step_is_valid", C.c_int),
        ("step_is_successful", C.c_int),
        ("reserved", C.c_int),
        ("cost", C.c_double),
        ("cost_change", C.c_double),
        ("gradient_max_norm", C.c_double),
        ("step_norm", C.c_double),
        ("relative_decrease", C.c_double),
        ("trust_region_radius", C.c_double),
    ]


class LmSummary(C.Structure):
    _fields_ = [
        ("termination", C.c_int),
        ("num_iterations", C.c_int),
        ("num_successful_steps", C.c_int),
        ("num_unsuccessful_steps", C.c_int),
        ("num_sweeps", C.c_int),
        ("reserved", C.c_int),
        ("initial_cost", C.c_double),
        ("final_cost", C.c_double),
        ("device_ms", C.c_double),
    ]


TERMINATION = {
    0: "RUNNING",
    1: "CONVERGENCE_FUNCTION",
    2: "CONVERGENCE_PARAMETER",
    3: "CONVERGENCE_GRADIENT",
    4: "CONVERGENCE_MIN_RADIUS",
    5: "NO_CONVERGENCE",
    6: "FAILURE",
}

# every symbol include/clc_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "clc_last_error": (C.c_char_p, []),
    "clc_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "clc_lm_default_options": (None, [C.POINTER(LmOptions)]),
    "clc_problem_create": (C.c_int, [C.POINTER(_P), C.POINTER(ProblemDesc)]),
    "clc_problem_create_gather": (C.c_int, [C.POINTER(_P), C.POINTER(GatherDesc)]),
    "clc_problem_create_synthetic": (C.c_int, [C.POINTER(_P), C.POINTER(SyntheticDesc)]),
    "clc_group_create_gather": (C.c_int, [C.POINTER(_P), C.POINTER(GatherDesc), C.POINTER(C.c_int), C.c_int]),
    "clc_group_create_synthetic": (C.c_int, [C.POINTER(_P), C.POINTER(SyntheticDesc), C.POINTER(C.c_int), C.c_int]),
    "clc_group_destroy": (C.c_int, [_P]),
    "clc_group_size": (C.c_int, [_P, C.POINTER(C.c_int), c_int64_p, c_int64_p]),
    "clc_group_problem": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "clc_group_eval": (C.c_int, [_P, c_double_p, c_double_p, c_double_p, c_double_p]),
    "clc_group_solve_lm": (C.c_int, [_P, c_double_p, C.POINTER(LmOptions), C.POINTER(LmSummary), C.POINTER(LmIteration), C.c_int]),
    "clc_group_information": (C.c_int, [_P, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "clc_group_closed_form": (C.c_int, [_P, c_double_p, C.POINTER(C.c_int), c_double_p, c_double_p]),
    "clc_default_devices": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]),
    "clc_upload_last_stats": (C.c_int, [c_double_p, c_double_p, c_int64_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "clc_problem_destroy": (C.c_int, [_P]),
    "clc_problem_sizes": (C.c_int, [_P, c_int64_p, c_int64_p, C.POINTER(C.c_int)]),
    "clc_problem_download": (C.c_int, [_P, c_double_p, c_int64_p, c_double_p, c_double_p, c_double_p]),
    "clc_problem_download_true_poses": (C.c_int, [_P, c_double_p]),
    "clc_eval": (C.c_int, [_P, c_double_p, c_double_p, c_double_p, c_double_p]),
    "clc_solve_lm": (C.c_int, [_P, c_double_p, C.POINTER(LmOptions), C.POINTER(LmSummary), C.POINTER(LmIteration), C.c_int]),
    "clc_information": (C.c_int, [_P, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "clc_closed_form": (C.c_int, [_P, c_double_p, C.POINTER(C.c_int), c_double_p, c_double_p]),
    "clc_problem_line_fit": (C.c_int, [_P, c_double_p, C.c_int, c_double_p]),
    "clc_line_fit_points": (C.c_int, [c_double_p, C.c_int64, c_double_p, C.c_int]),
    "clc_scan_segments": (C.c_int, [C.POINTER(C.c_float), C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_double,
                                    C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int]),
    "clc_problems_create_from_scans": (C.c_int, [C.POINTER(ScanDesc), C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int32),
                                                 c_double_p]),
    "clc_scan_last_stats": (C.c_int, [C.POINTER(C.c_float), c_int64_p, c_int64_p]),
    "clc_estimate_board_poses": (C.c_int, [C.POINTER(CameraDesc), C.c_int64, c_int64_p, C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                           c_double_p, C.POINTER(C.c_int32), C.c_int]),
    "clc_T_to_pose7": (None, [c_double_p, c_double_p]),
    "clc_pose7_to_T": (None, [c_double_p, c_double_p]),
    "clc_shard_range": (C.c_int, [C.c_int64, c_int64_p, C.c_int, C.c_int, c_int64_p, c_int64_p]),
    "clc_comm_unique_id": (C.c_int, [_P]),
    "clc_comm_create": (C.c_int, [C.POINTER(_P), _P, C.c_int, C.c_int, C.c_int]),
    "clc_comm_destroy": (C.c_int, [_P]),
    "clc_comm_p2p_export": (C.c_int, [_P, _P]),
    "clc_comm_p2p_import": (C.c_int, [_P, _P]),
    "clc_problem_attach_comm": (C.c_int, [_P, _P]),
    "clc_problem_set_allreduce_mode": (C.c_int, [_P, C.c_int]),
    "clc_bench_eval": (C.c_int, [_P, c_double_p, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "clc_problem_algorithmic_bytes": (C.c_int, [_P, c_int64_p]),
    "clc_problem_streamed_bytes": (C.c_int, [_P, c_int64_p]),
    "clc_problem_set_planar_mode": (C.c_int, [_P, C.c_int]),
    "clc_debug_pack": (C.c_int, [C.c_int64, C.POINTER(c_double_p), c_int64_p, C.c_int64, C.c_int64, C.c_int, c_double_p,
                                 C.POINTER(C.c_int)]),
    "clc_bench_h2d": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "clc_solve_readback_bytes": (C.c_int64, []),
    "clc_host_alloc": (C.c_int, [C.POINTER(_P), C.c_int64]),
    "clc_host_free": (C.c_int, [_P]),
    "clc_launch_count": (C.c_int64, []),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load():
    """dlopen libclc_b200.so (building it first when nvcc is present and the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("CLC_LIB_PATH", _build.LIB_PATH)  # CLC_LIB_PATH: load an experimental build variant
    if path == _build.LIB_PATH and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: use the prebuilt file if there is one
            if not os.path.exists(path):
                raise ClcError(f"libclc_b200.so is missing and cannot be built: {exc}") from exc
    try:
        L = C.CDLL(path)
    except OSError as exc:
        raise ClcError(f"cannot load {path}: {exc}") from exc
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        msg = load().clc_last_error()
        raise ClcError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")
