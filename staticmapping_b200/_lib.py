"""ctypes loader for libsm_b200.so (the C ABI declared in include/sm_b200.h).

There is NO CPU fallback: if the shared library is missing, or no CUDA device is visible
when a matcher is created, this raises.  (The library itself loads on a CPU-only box so
that the symbol table can be checked there.)"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SM_B200_LIB: A/B builds for profiles/ (same ABI); the product library is libsm_b200.so
LIB_PATH = os.environ.get("SM_B200_LIB") or os.path.join(_HERE, "libsm_b200.so")


class AlignInfo(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("status", C.c_int32), ("solve_path", C.c_int32),
                ("reserved", C.c_int32), ("kept", C.c_int64), ("limit", C.c_double),
                ("ms_upload", C.c_float), ("ms_prologue", C.c_float),
                ("ms_iterations", C.c_float), ("kernel_launches", C.c_int32),
                ("ms_knn", C.c_float), ("ms_accum", C.c_float), ("ms_finish", C.c_float),
                ("profiled_iterations", C.c_int32), ("evaluations", C.c_int32),
                ("trans_probability", C.c_double), ("mean_neighbors", C.c_double),
                ("aux", C.c_double * 4)]


class Pair(C.Structure):
    _fields_ = [("source", C.c_void_p), ("n_source", C.c_int64), ("target", C.c_void_p),
                ("target_normals", C.c_void_p), ("n_target", C.c_int64), ("guess", C.c_void_p),
                ("on_device", C.c_int32), ("reserved", C.c_int32)]


_lib = None

_DP = C.POINTER(C.c_double)
_IP = C.POINTER(C.c_int32)
_VP = C.c_void_p

# name -> (restype, argtypes); this table must list every symbol of include/sm_b200.h
SIGNATURES = {
    "sm_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_VP)]),
    "sm_destroy": (C.c_int, [_VP]),
    "sm_set_option": (C.c_int, [_VP, C.c_char_p, C.c_char_p]),
    "sm_print_options": (C.c_int, [_VP, C.c_char_p, C.c_int64]),
    "sm_get_type": (C.c_int, [_VP]),
    "sm_set_input_source": (C.c_int, [_VP, _VP, C.c_int64]),
    "sm_set_input_target": (C.c_int, [_VP, _VP, _VP, C.c_int64]),
    "sm_set_input_source_f32": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64]),
    "sm_set_input_target_f32": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64]),
    "sm_set_input_source_f32_device": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64]),
    "sm_set_input_target_f32_device": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64]),
    "sm_set_input_source_device": (C.c_int, [_VP, _VP, C.c_int64]),
    "sm_set_input_target_device": (C.c_int, [_VP, _VP, _VP, C.c_int64]),
    "sm_align": (C.c_int, [_VP, _DP, _DP]),
    "sm_align_async": (C.c_int, [_VP, _DP]),
    "sm_align_wait": (C.c_int, [_VP, _DP]),
    "sm_align_batch": (C.c_int, [_VP, C.c_int32, _VP, _VP, _VP]),
    "sm_align_pairs": (C.c_int, [_VP, C.c_int32, _VP, C.c_int32, _VP, _VP, _VP]),
    "sm_get_fitness_score": (C.c_double, [_VP]),
    "sm_get_align_info": (C.c_int, [_VP, C.POINTER(AlignInfo)]),
    "sm_set_stream": (C.c_int, [_VP, _VP]),
    "sm_last_error": (C.c_char_p, [_VP]),
    "sm_knn1": (C.c_int, [C.c_int, _VP, C.c_int64, _VP, C.c_int64, C.c_double, C.c_int, _VP, _VP]),
    "sm_calculate_normals": (C.c_int, [C.c_int, _VP, C.c_int64, _VP, _VP, C.POINTER(C.c_int64)]),
    "sm_motion_compensation": (C.c_int, [C.c_int, _VP, C.c_int64, C.c_int64, _DP, _VP]),
    "sm_motion_compensation_device": (C.c_int, [C.c_int, _VP, C.c_int64, C.c_int64, _DP, _VP, _VP]),
    "sm_voxel_grid_filter": (C.c_int, [C.c_int, _VP, C.c_int64, C.c_int64, C.c_float, _VP, C.POINTER(C.c_int64)]),
    "sm_m2dp_descriptor_length": (C.c_int64, [C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_int32]),
    "sm_m2dp": (C.c_int, [C.c_int, _VP, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_int32,
                          _VP, C.c_int64, _VP]),
    "sm_m2dp_match": (C.c_double, [_VP, _VP, C.c_int64]),
    "sm_mrvm_create": (C.c_int, [C.c_int, _VP, C.c_int64, C.POINTER(_VP)]),
    "sm_mrvm_destroy": (C.c_int, [_VP]),
    "sm_mrvm_set_offset_z": (C.c_int, [_VP, C.c_float]),
    "sm_mrvm_insert": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _VP]),
    "sm_mrvm_insert_device": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _VP, _VP]),
    "sm_mrvm_size": (C.c_int64, [_VP]),
    "sm_mrvm_output": (C.c_int, [_VP, C.c_float, C.c_int32, _VP, C.c_int64, C.POINTER(C.c_int64)]),
    "sm_mrvm_phase_ms": (C.c_int, [_VP, _VP]),
    "sm_filter_chain_create": (C.c_int, [C.c_int, C.POINTER(_VP)]),
    "sm_filter_chain_destroy": (C.c_int, [_VP]),
    "sm_filter_chain_add": (C.c_int, [_VP, C.c_char_p]),
    "sm_filter_chain_set_param": (C.c_int, [_VP, C.c_int32, C.c_char_p, C.c_int32, C.c_char_p]),
    "sm_filter_chain_valid": (C.c_int, [_VP, C.c_int32]),
    "sm_filter_chain_set_seed": (C.c_int, [_VP, C.c_uint64]),
    "sm_filter_chain_filter": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _VP, C.c_int64, C.POINTER(C.c_int64), _VP]),
    "sm_filter_chain_filter_device": (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _VP, C.c_int64, C.POINTER(C.c_int64),
                                                _VP, _VP]),
    "sm_filter_chain_stage_counts": (C.c_int, [_VP, _VP, C.c_int32]),
    "sm_filter_chain_stage_ms": (C.c_int, [_VP, _VP, C.c_int32]),
    # include/sm_b200_debug.h (test hooks)
    "sm_debug_solve6": (C.c_int, [C.c_int, _VP, _VP, _VP, _VP]),
    "sm_debug_solve6_host": (C.c_int, [_VP, _VP, _VP, _VP]),
    "sm_debug_bfgs_minimize": (C.c_int, [_VP, _VP, _VP, C.c_double, C.c_int32, _VP, _VP, _VP]),
    "sm_debug_ndt_newton": (C.c_int, [_VP, _VP, _VP, C.c_int32, C.c_float, C.c_double, C.c_double, C.c_double, C.c_int32,
                                      _VP, _VP, _VP, _VP]),
    "sm_debug_normals_leaf": (C.c_int, [_VP, C.c_int32, _VP, _VP, _VP]),
    "sm_debug_voxel_index": (C.c_int, [C.c_int32, _VP, C.c_float, C.c_int32, _VP]),
    "sm_debug_gicp_point": (C.c_int, [C.c_int32, _VP, _VP]),
    "sm_debug_gicp_outer": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "sm_debug_gicp_host": (C.c_int, [C.c_int32, _VP, _VP]),
    "sm_debug_motion_host": (C.c_int, [_VP, C.c_int64, _DP, _VP]),
    "sm_debug_icp_host": (C.c_int, [C.c_int32, _VP, C.c_int64, _VP]),
    "sm_debug_ndt_leaf": (C.c_int, [_VP, C.c_int32, C.c_int32, C.c_double, _VP, _VP, _VP, _VP, _VP]),
    "sm_debug_ndt_term": (C.c_int, [_VP, C.c_double, C.c_float, C.c_int32, _VP, _VP, _VP, _VP, _VP]),
    "sm_debug_ndt_host": (C.c_int, [C.c_int32, _VP, _VP]),
    "sm_debug_mrvm_ray": (C.c_int, [_VP, _VP, C.c_float, _VP, C.c_int64, C.POINTER(C.c_int64)]),
    "sm_debug_mrvm_update": (C.c_int, [C.c_float, C.c_float, _VP, _VP, _VP, C.c_int64, _VP, _VP]),
    "sm_debug_mrvm_state": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_int64, C.POINTER(C.c_int64)]),
    "sm_debug_filter_points": (C.c_int, [C.c_int32, _VP, C.c_int64, C.c_int64, _VP, _VP]),
    "sm_debug_filter_fit_lines": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int64, C.POINTER(C.c_int64)]),
    "sm_debug_filter_line_fit": (C.c_int, [_VP, C.c_int64, _VP]),
    "sm_debug_knn1_batched": (C.c_int, [C.c_int, _VP, C.c_int64, _VP, C.c_int64, C.c_double, C.c_int, C.c_int32, _VP, _VP]),
    "sm_device_count": (C.c_int, []),
    "sm_version": (C.c_char_p, []),
}


def lib():
    """Load libsm_b200.so; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (nvcc, sm_100a).  staticmapping_b200 has no CPU fallback.")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib
