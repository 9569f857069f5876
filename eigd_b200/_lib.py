"""ctypes binding of libeigd_b200.so (the C-ABI declared in include/eigd_b200.h).

The product path has no CPU fallback: if the shared library is missing the import of any
compute entry point raises, and if no CUDA device is visible the first device call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libeigd_b200.so")

c_int = ctypes.c_int
c_i64 = ctypes.c_int64
c_dbl = ctypes.c_double
c_ptr = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/eigd_b200.h one to one
SIGNATURES = {
    "eigd_version": (c_int, []),
    "eigd_last_error": (ctypes.c_char_p, []),
    "eigd_device_count": (c_int, [c_ptr]),
    "eigd_set_stream": (c_int, [c_ptr]),
    "eigd_launch_count": (c_i64, []),
    "eigd_csr_spmm": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_int, c_dbl, c_dbl]),
    "eigd_axpby": (c_int, [c_i64, c_dbl, c_ptr, c_dbl, c_ptr, c_ptr]),
    "eigd_gemm_tn_workspace": (c_i64, [c_int, c_int]),
    "eigd_gemm_tn": (c_int, [c_i64, c_int, c_int, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_int, c_ptr]),
    "eigd_gemm_nn": (c_int, [c_i64, c_int, c_int, c_dbl, c_ptr, c_i64, c_i64, c_ptr, c_int, c_dbl, c_ptr, c_i64, c_i64]),
    "eigd_col_dot": (c_int, [c_i64, c_int, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "eigd_col_axpy": (c_int, [c_i64, c_int, c_dbl, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64]),
    "eigd_mgs_sweep": (c_int, [c_i64, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_col_scale": (c_int, [c_i64, c_int, c_int, c_ptr, c_ptr, c_i64, c_i64]),
    "eigd_copy2d": (c_int, [c_i64, c_int, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64]),
    "eigd_symbolic_create": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr, c_ptr]),
    "eigd_symbolic_destroy": (None, [c_ptr]),
    "eigd_symbolic_query": (c_i64, [c_ptr, c_int]),
    "eigd_symbolic_get": (c_i64, [c_ptr, c_int, c_ptr, c_i64]),
    "eigd_symbolic_assembly_map_host": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr]),
    "eigd_symbolic_assembly_map_device": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr]),
    "eigd_solve_plan_get": (c_i64, [c_ptr, c_int, c_int, c_int, c_int, c_ptr, c_i64]),
    "eigd_factor_create": (c_int, [c_ptr, c_int, c_ptr]),
    "eigd_factor_workspace_bytes": (c_i64, [c_ptr, c_int]),
    "eigd_factor_create_in": (c_int, [c_ptr, c_int, c_ptr, c_i64, c_ptr]),
    "eigd_factor_workspace_bytes_fronts": (c_i64, [c_ptr, c_int, c_int]),
    "eigd_factor_create_in_fronts": (c_int, [c_ptr, c_int, c_int, c_ptr, c_i64, c_ptr]),
    "eigd_factor_destroy": (None, [c_ptr]),
    "eigd_factor_numeric": (c_int, [c_ptr, c_i64, c_ptr, c_ptr]),
    "eigd_factor_numeric_pool": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64]),
    "eigd_factor_info": (c_int, [c_ptr, c_ptr]),
    "eigd_factor_set_pivoting": (c_int, [c_ptr, c_int]),
    "eigd_factor_pivot_counts": (c_int, [c_ptr, c_ptr]),
    "eigd_dmma_peak": (c_int, [c_int, c_int, c_ptr]),
    "eigd_factor_solve": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_int]),
    "eigd_factor_set_refinement": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_int]),
    "eigd_factor_apply": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_int]),
    "eigd_factor_bytes": (c_i64, [c_ptr]),
    "eigd_solve_timing_begin": (c_int, []),
    "eigd_solve_timing_end": (c_int, [c_ptr, c_ptr]),
    "eigd_solve_set_phase_times": (c_int, [c_ptr]),
    "eigd_solve_set_trace": (c_int, [c_ptr]),
    "eigd_solve_set_skew": (c_int, [c_ptr]),
    "eigd_solve_num_phases": (c_int, [c_ptr]),
    "eigd_lanczos_extend": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_ptr, c_ptr, c_ptr,
                                    c_ptr, c_int, c_ptr]),
    "eigd_stored_assemble": (c_int, [c_i64, c_ptr, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_stored_quadform": (c_int, [c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_i64, c_ptr, c_ptr,
                                     c_ptr, c_ptr, c_dbl, c_dbl]),
    "eigd_segment_sum": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_dbl, c_ptr]),
    "eigd_block_lanczos_extend": (c_int, [c_ptr, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int,
                                          c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_block_lanczos_start": (c_int, [c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "eigd_q4_assemble": (c_int, [c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "eigd_q4_quadforms": (c_int, [c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr, c_ptr, c_dbl, c_dbl, c_ptr]),
    "eigd_q4_material": (c_int, [c_int, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_h8_element_matrices": (c_int, [c_int, c_ptr, c_ptr, c_dbl, c_dbl, c_dbl, c_ptr, c_ptr]),
    "eigd_h8_thermal_element_matrices": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_t10_element_matrices": (c_int, [c_int, c_ptr, c_ptr, c_dbl, c_dbl, c_dbl, c_ptr, c_ptr]),
    "eigd_t10_thermal_element_matrices": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_h8_stress_stiffness": (c_int, [c_int, c_ptr, c_ptr, c_dbl, c_dbl, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_h8_gderiv_u": (c_int, [c_int, c_ptr, c_ptr, c_dbl, c_dbl, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_i64, c_ptr]),
    "eigd_node_gather": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_dbl, c_ptr]),
    "eigd_dof_gather": (c_int, [c_int, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_filter_project": (c_int, [c_int, c_dbl, c_dbl, c_ptr, c_ptr, c_ptr]),
    "eigd_q4_stress": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "eigd_q4_assemble_geometric": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr]),
    "eigd_q4_gderiv": (c_int, [c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr, c_ptr, c_ptr, c_dbl, c_ptr, c_ptr]),
    "eigd_expand_rows": (c_int, [c_i64, c_int, c_ptr, c_ptr, c_ptr]),
    "eigd_reduce_rows": (c_int, [c_i64, c_int, c_ptr, c_ptr, c_ptr]),
}

_lib = None


class EigdNativeError(RuntimeError):
    pass


def load():
    """Load the shared library (built by build.sh / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise EigdNativeError(
            "eigd_b200: %s is missing -- run ./build.sh (there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().eigd_last_error()
        raise EigdNativeError("eigd_b200 %s failed (rc=%d): %s" % (what, rc, (msg or b"").decode()))
