"""ctypes loader for the C-ABI library sim3opt_b200/lib/libsim3opt_b200.so.

The library is built in-tree by ``__graft_entry__.build()`` (or ``make -C sim3opt_b200/csrc``).
There is no Python/CPU fallback: if the shared object is missing, loading fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsim3opt_b200.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_up = C.POINTER(C.c_uint8)


class Stats(C.Structure):
    _fields_ = [
        ("ms_linearize", C.c_double), ("ms_solve", C.c_double), ("ms_chi2", C.c_double),
        ("ms_update", C.c_double), ("ms_total", C.c_double),
        ("kernel_launches", C.c_int64), ("pcg_iterations", C.c_int64),
        ("lm_iterations", C.c_int64), ("lm_trials", C.c_int64),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("n_vertices", C.c_int32), ("n_free", C.c_int32), ("n_edges", C.c_int32),
        ("n_blocks", C.c_int32), ("dim", C.c_int32),
        ("ms_spmv_sampled", C.c_double), ("n_spmv_sampled", C.c_int64),
        ("multilevel_levels", C.c_int32), ("p2p_halo", C.c_int32),
        ("direct_solves", C.c_int64), ("direct_levels", C.c_int32), ("direct_blocks", C.c_int32),
        ("pcg_unconverged", C.c_int64),
        ("sum_ms_linearize", C.c_double), ("sum_ms_solve", C.c_double), ("sum_ms_update", C.c_double),
        ("last_step_inf", C.c_double), ("est_distance", C.c_double),
        ("stop_reason", C.c_int32), ("reserved0", C.c_int32),
        ("multilevel_rebuilds", C.c_int64), ("multilevel_reuses", C.c_int64),
    ]


# every symbol include/sim3opt_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "s3o_last_error": (C.c_char_p, []),
    "s3o_version": (C.c_int, []),
    "s3o_device_count": (C.c_int, []),
    "s3o_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "s3o_destroy": (C.c_int, [C.c_void_p]),
    "s3o_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "s3o_comm_unique_id": (C.c_int, [C.c_char_p]),
    "s3o_set_comm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "s3o_host_partition": (C.c_int, [C.c_int, _up, C.c_int, _ip, _ip, C.c_int, C.c_int, _ip, _ip, _ip, _ip, _ip, _ip, _ip, _ip]),
    "s3o_set_vertices": (C.c_int, [C.c_void_p, C.c_int, _dp, _up, _dp]),
    "s3o_set_edges": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp, _dp]),
    "s3o_add_vertices": (C.c_int, [C.c_void_p, C.c_int, _dp, _up, _dp]),
    "s3o_add_edges": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp, _dp]),
    "s3o_set_estimates": (C.c_int, [C.c_void_p, _dp]),
    "s3o_set_robust": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "s3o_set_jacobian_mode": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "s3o_set_math_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "s3o_set_scale_model": (C.c_int, [C.c_void_p, C.c_int]),
    "s3o_set_lm": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_int]),
    "s3o_set_stop_rules": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "s3o_set_pcg": (C.c_int, [C.c_void_p, C.c_double, C.c_int]),
    "s3o_set_preconditioner": (C.c_int, [C.c_void_p, C.c_int]),
    "s3o_set_linear_solver": (C.c_int, [C.c_void_p, C.c_int]),
    "s3o_build_structure": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "s3o_host_structure": (C.c_int, [C.c_int, _up, C.c_int, _ip, _ip, C.POINTER(C.c_int), C.POINTER(C.c_int), _ip, _ip, _ip]),
    "s3o_host_multilevel": (C.c_int, [C.c_int, _up, C.c_int, _ip, _ip, C.c_int, C.c_int, C.POINTER(C.c_int), _ip, _ip, _ip]),
    "s3o_host_direct_plan": (C.c_int, [C.c_int, _up, C.c_int, _ip, _ip, C.c_int64, C.POINTER(C.c_int64), _ip, _ip, _ip, _ip, _ip, _ip, _ip, _ip]),
    "s3o_align_similarity": (C.c_int, [C.c_int, C.c_int, _dp, _dp, C.c_int, _dp, _dp, _dp]),
    "s3o_get_structure": (C.c_int, [C.c_void_p, _ip, _ip]),
    "s3o_get_hessian_index": (C.c_int, [C.c_void_p, _ip]),
    "s3o_chi2": (C.c_int, [C.c_void_p, _dp]),
    "s3o_edge_errors": (C.c_int, [C.c_void_p, _dp]),
    "s3o_linearize": (C.c_int, [C.c_void_p]),
    "s3o_get_hessian": (C.c_int, [C.c_void_p, _dp, _dp]),
    "s3o_max_diag": (C.c_int, [C.c_void_p, _dp]),
    "s3o_solve": (C.c_int, [C.c_void_p, C.c_double, _dp, C.POINTER(C.c_int), _dp]),
    "s3o_hessian_multiply": (C.c_int, [C.c_void_p, C.c_double, _dp, _dp]),
    "s3o_update": (C.c_int, [C.c_void_p, _dp]),
    "s3o_multilevel_prepare": (C.c_int, [C.c_void_p, C.c_double, _ip, C.c_int]),
    "s3o_get_multilevel_level": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _ip, _ip, _dp, _dp, _dp]),
    "s3o_get_multilevel_coarsest_inverse": (C.c_int, [C.c_void_p, _dp]),
    "s3o_apply_preconditioner": (C.c_int, [C.c_void_p, C.c_double, _dp, _dp]),
    "s3o_direct_schedule": (C.c_int, [C.c_void_p, _ip, C.c_int]),
    "s3o_get_direct_factor": (C.c_int, [C.c_void_p, _dp, _dp]),
    "s3o_smallest_eigenvector": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp, _dp, _dp, C.POINTER(C.c_int)]),
    "s3o_compute_marginals": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp]),
    "s3o_optimize": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.POINTER(C.c_int), _dp, _dp, _dp, C.c_int]),
    "s3o_get_vertices": (C.c_int, [C.c_void_p, _dp]),
    "s3o_estimate_slice": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "s3o_set_estimates_slice": (C.c_int, [C.c_void_p, _dp]),
    "s3o_get_vertices_slice": (C.c_int, [C.c_void_p, _dp]),
    "s3o_set_lm_resume": (C.c_int, [C.c_void_p, C.c_int]),
    "s3o_snapshot_estimates": (C.c_int, [C.c_void_p]),
    "s3o_restore_estimates": (C.c_int, [C.c_void_p]),
    "s3o_ba_set_cameras": (C.c_int, [C.c_void_p, C.c_int, _dp, _up]),
    "s3o_ba_set_points": (C.c_int, [C.c_void_p, C.c_int, _dp, _up]),
    "s3o_ba_set_observations": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp, _dp]),
    "s3o_ba_set_intrinsics": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "s3o_ba_set_estimates": (C.c_int, [C.c_void_p, _dp, _dp]),
    "s3o_ba_get_cameras": (C.c_int, [C.c_void_p, _dp]),
    "s3o_ba_get_points": (C.c_int, [C.c_void_p, _dp]),
    "s3o_ba_get_sizes": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "s3o_ba_edge_errors": (C.c_int, [C.c_void_p, _dp]),
    "s3o_ba_get_system": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _dp]),
    "s3o_ba_get_schur": (C.c_int, [C.c_void_p, C.c_double, _dp, _dp]),
    "s3o_ba_compute_marginals": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp]),
    "s3o_linsolver_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "s3o_linsolver_destroy": (C.c_int, [C.c_void_p]),
    "s3o_linsolver_solve": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp, C.c_int, C.c_double, _dp, _dp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "s3o_linsolver_solve_pattern": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _dp, C.c_int, C.c_int, _ip, _ip, _dp]),
    "s3o_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "s3o_reset_stats": (C.c_int, [C.c_void_p]),
    "s3o_estimate_sigma_squared": (C.c_int, [C.c_void_p, C.c_int, _dp]),
}

_lib = None


def load():
    """dlopen the library and bind every declared symbol (raises if one is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C sim3opt_b200/csrc` (the CUDA extension is mandatory; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib
