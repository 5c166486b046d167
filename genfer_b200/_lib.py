"""ctypes loader for libgenfer_taylor.so (the C ABI declared in include/genfer_taylor.h).

The library must have been built in-tree (``python genfer_b200/build.py`` or
``__graft_entry__.build()``).  Loading fails loudly if it is missing -- there is no Python or CPU
fallback for the f64 path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgenfer_taylor.so")
UNBOUNDED = 2**64 - 1
MAX_NDIM = 24

STATUS = {0: "GTP_OK", 1: "GTP_ERR_INDEX", 2: "GTP_ERR_SHAPE", 3: "GTP_ERR_OOM", 4: "GTP_ERR_CUDA", 5: "GTP_ERR_ARG"}

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
f64p = C.POINTER(C.c_double)
vp = C.c_void_p
vpp = C.POINTER(C.c_void_p)
intp = C.POINTER(C.c_int)

_SIGS = {
    # name: (restype, argtypes)
    "gtp_ctx_create": (C.c_int, [C.c_int, vp, vpp]),
    "gtp_ctx_destroy": (None, [vp]),
    "gtp_last_error": (C.c_char_p, [vp]),
    "gtp_ctx_synchronize": (C.c_int, [vp]),
    "gtp_ctx_trim": (C.c_int, [vp]),
    "gtp_ctx_stream": (vp, [vp]),
    "gtp_ctx_launch_count": (C.c_uint64, [vp]),
    "gtp_ctx_set_fast_mul": (C.c_int, [vp, C.c_int]),
    "gtp_nccl_unique_id": (C.c_int, [vp]),
    "gtp_ctx_create_group": (C.c_int, [C.c_int, vp, C.c_int, C.c_int, vp, vpp]),
    "gtp_ctx_group_info": (C.c_int, [vp, intp, intp, u64p, u64p]),
    "gtp_ctx_set_partition_threshold": (C.c_int, [vp, C.c_uint64]),
    "gtp_partition_rows": (C.c_uint64, [C.c_uint64, C.c_int, C.c_int, u64p]),
    "gtp_partition_block": (None, [C.c_uint64, C.c_int, C.c_int, u64p, u64p, u64p]),
    "gtp_from_host_block": (C.c_int, [vp, C.c_int, u64p, u64p, vp, vpp]),
    "gtp_from_device_block": (C.c_int, [vp, C.c_int, u64p, u64p, vp, vpp]),
    "gtp_is_distributed": (C.c_int, [vp]),
    "gtp_replicate": (C.c_int, [vp, vp]),
    "gtp_local_rows": (C.c_uint64, [vp, u64p]),
    "gtp_to_host_local": (C.c_int, [vp, vp, vp]),
    "gtp_from_host": (C.c_int, [vp, C.c_int, u64p, u64p, f64p, vpp]),
    "gtp_from_device": (C.c_int, [vp, C.c_int, u64p, u64p, vp, vpp]),
    "gtp_to_host": (C.c_int, [vp, vp, vp]),
    "gtp_device_ptr": (C.c_int, [vp, vp, vpp]),
    "gtp_clone": (C.c_int, [vp, vp, vpp]),
    "gtp_free": (None, [vp, vp]),
    "gtp_ndim": (C.c_int, [vp]),
    "gtp_len": (C.c_uint64, [vp]),
    "gtp_shape": (None, [vp, u64p]),
    "gtp_degrees_p1": (None, [vp, u64p]),
    "gtp_from_scalar": (C.c_int, [vp, C.c_double, vpp]),
    "gtp_zero_with": (C.c_int, [vp, C.c_int, u64p, vpp]),
    "gtp_var": (C.c_int, [vp, C.c_uint64, C.c_double, C.c_uint64, vpp]),
    "gtp_var_at_zero": (C.c_int, [vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_var_with_degrees_p1": (C.c_int, [vp, C.c_uint64, C.c_double, C.c_int, u64p, vpp]),
    "gtp_add": (C.c_int, [vp, vp, vp, vpp]),
    "gtp_sub": (C.c_int, [vp, vp, vp, vpp]),
    "gtp_mul": (C.c_int, [vp, vp, vp, vpp]),
    "gtp_div": (C.c_int, [vp, vp, vp, vpp]),
    "gtp_neg": (C.c_int, [vp, vp, vpp]),
    "gtp_exp": (C.c_int, [vp, vp, vpp]),
    "gtp_log": (C.c_int, [vp, vp, vpp]),
    "gtp_pow": (C.c_int, [vp, vp, C.c_uint32, vpp]),
    "gtp_derivative": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_taylor_expansion_of_coeff": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_shift_down": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_coefficients_of_term": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_taylor_polynomial": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_taylor_polynomial_terms": (C.c_int, [vp, vp, C.c_uint64, u64p, C.c_int, vpp]),
    "gtp_subst_var": (C.c_int, [vp, vp, C.c_uint64, vp, vpp]),
    "gtp_truncate_to_degree_p1": (C.c_int, [vp, vp, C.c_uint64, vpp]),
    "gtp_remove_last_variable": (C.c_int, [vp, vp, vpp]),
    "gtp_extend_to_dim": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gtp_extend": (C.c_int, [vp, vp, C.c_int, u64p, vpp]),
    "gtp_constant_term": (C.c_int, [vp, vp, f64p]),
    "gtp_coefficient": (C.c_int, [vp, vp, u64p, C.c_int, f64p]),
    "gtp_gather_axis": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, f64p]),
    "gtp_extract_constant": (C.c_int, [vp, vp, intp, f64p]),
    "gtp_extract_linear": (C.c_int, [vp, vp, intp, f64p, f64p, u64p]),
    "gtp_is_zero": (C.c_int, [vp, vp, intp]),
    "gtp_is_one": (C.c_int, [vp, vp, intp]),
    "gtp_evaluate_all_one": (C.c_int, [vp, vp, f64p]),
    "gtp_eq": (C.c_int, [vp, vp, vp, intp]),
    "gtp_mul_rows_raw": (C.c_int, [vp, C.c_int, u64p, vp, u64p, vp, u64p, C.c_uint64, C.c_uint64, C.c_uint64, vp]),
    "gtp_mul_rowlist_raw": (C.c_int, [vp, C.c_int, u64p, vp, u64p, vp, u64p, u64p, C.c_uint64, vp]),
    "gtp_mul_macs": (C.c_double, [C.c_int, u64p, u64p, u64p]),
    "gtp_mul_kernel_kind": (C.c_int, [vp, C.c_int, u64p, u64p, u64p]),
    "gtp_fp64_peak_probe": (C.c_int, [vp, C.c_int, C.c_int, f64p, f64p]),
    "gtp_run_sgcl": (C.c_int, [vp, C.c_char_p, C.c_int64, C.c_int, C.c_uint64, vpp, C.c_char_p, C.c_size_t]),
    "gtp_sgcl_free": (None, [vp]),
    "gtp_sgcl_report": (C.c_char_p, [vp]),
    "gtp_sgcl_moments": (None, [vp, f64p]),
    "gtp_sgcl_limit": (C.c_uint64, [vp]),
    "gtp_sgcl_is_normalized": (C.c_int, [vp]),
    "gtp_sgcl_probs": (None, [vp, f64p, f64p]),
    "gtp_sgcl_stats": (None, [vp, u64p, u64p]),
    "gtp_sgcl_moment_bounds": (None, [vp, f64p]),
    "gtp_sgcl_prob_bounds": (None, [vp, f64p, f64p]),
    "gtp_run_sgcl_bounds": (C.c_int, [vp, C.c_char_p, C.c_int64, C.c_uint64, f64p, f64p, C.c_char_p, C.c_size_t]),
    "gti_from_scalar": (C.c_int, [vp, C.c_double, C.c_double, vpp]),
    "gti_zero_with": (C.c_int, [vp, C.c_int, u64p, vpp]),
    "gti_var": (C.c_int, [vp, C.c_uint64, C.c_double, C.c_double, C.c_uint64, vpp]),
    "gti_var_at_zero": (C.c_int, [vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_var_with_degrees_p1": (C.c_int, [vp, C.c_uint64, C.c_double, C.c_double, C.c_int, u64p, vpp]),
    "gti_from_host": (C.c_int, [vp, C.c_int, u64p, u64p, vp, C.c_int, vpp]),
    "gti_to_host": (C.c_int, [vp, vp, vp]),
    "gti_free": (None, [vp, vp]),
    "gti_ndim": (C.c_int, [vp]),
    "gti_len": (C.c_uint64, [vp]),
    "gti_shape": (None, [vp, u64p]),
    "gti_degrees_p1": (None, [vp, u64p]),
    "gti_add": (C.c_int, [vp, vp, vp, vpp]),
    "gti_sub": (C.c_int, [vp, vp, vp, vpp]),
    "gti_mul": (C.c_int, [vp, vp, vp, vpp]),
    "gti_div": (C.c_int, [vp, vp, vp, vpp]),
    "gti_neg": (C.c_int, [vp, vp, vpp]),
    "gti_exp": (C.c_int, [vp, vp, vpp]),
    "gti_log": (C.c_int, [vp, vp, vpp]),
    "gti_pow": (C.c_int, [vp, vp, C.c_uint32, vpp]),
    "gti_derivative": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_taylor_expansion_of_coeff": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_shift_down": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_coefficients_of_term": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_taylor_polynomial_terms": (C.c_int, [vp, vp, C.c_uint64, u64p, C.c_int, vpp]),
    "gti_subst_var": (C.c_int, [vp, vp, C.c_uint64, vp, vpp]),
    "gti_truncate_to_degree_p1": (C.c_int, [vp, vp, C.c_uint64, vpp]),
    "gti_remove_last_variable": (C.c_int, [vp, vp, vpp]),
    "gti_extend_to_dim": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vpp]),
    "gti_constant_term": (C.c_int, [vp, vp, f64p]),
    "gti_extract_constant": (C.c_int, [vp, vp, intp, f64p]),
    "gti_gather_axis": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, vp]),
    "gtu_constant": (C.c_int, [vp, C.c_double, vpp]),
    "gtu_from_coefficients": (C.c_int, [vp, f64p, C.c_uint64, vpp]),
    "gtu_var": (C.c_int, [vp, C.c_double, C.c_uint64, vpp]),
    "gtu_free": (None, [vp, vp]),
    "gtu_is_constant": (C.c_int, [vp]),
    "gtu_order": (C.c_uint64, [vp]),
    "gtu_to_host": (C.c_int, [vp, vp, f64p]),
    "gtu_coeff": (C.c_int, [vp, vp, C.c_uint64, f64p]),
    "gtu_derivative": (C.c_int, [vp, vp, C.c_uint64, f64p]),
    "gtu_add": (C.c_int, [vp, vp, vp, vpp]),
    "gtu_sub": (C.c_int, [vp, vp, vp, vpp]),
    "gtu_mul": (C.c_int, [vp, vp, vp, vpp]),
    "gtu_div": (C.c_int, [vp, vp, vp, vpp]),
    "gtu_neg": (C.c_int, [vp, vp, vpp]),
    "gtu_exp": (C.c_int, [vp, vp, vpp]),
    "gtu_log": (C.c_int, [vp, vp, vpp]),
    "gtu_pow": (C.c_int, [vp, vp, C.c_uint32, vpp]),
    "gtu_subst": (C.c_int, [vp, vp, vp, vpp]),
    "gtu_taylor_expansion_of_coeff": (C.c_int, [vp, vp, C.c_uint64, vpp]),
    "gtu_eq": (C.c_int, [vp, vp, vp, intp]),
    "gtu_program_create": (C.c_int, [vp, vpp]),
    "gtu_program_free": (None, [vp, vp]),
    "gtu_program_constant": (C.c_int, [vp, vp, C.c_double, u32p]),
    "gtu_program_var": (C.c_int, [vp, vp, C.c_double, C.c_uint64, u32p]),
    "gtu_program_from_coefficients": (C.c_int, [vp, vp, f64p, C.c_uint64, u32p]),
    "gtu_program_op": (C.c_int, [vp, vp, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, u32p]),
    "gtu_program_slot": (C.c_int, [vp, C.c_uint32, intp, u64p]),
    "gtu_program_run": (C.c_int, [vp, vp, u32p, C.c_int, f64p]),
}

SYMBOLS = tuple(_SIGS)
_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python genfer_b200/build.py` "
                "(there is no CPU fallback for the f64 Taylor path)")
        if "GTP_NCCL_LIB" not in os.environ:
            # group contexts dlopen NCCL: in a Python process it must be the copy PyTorch is linked against (same soname,
            # the loader would otherwise hand torch the system's older libnccl.so.2 -- or us torch's, depending on order)
            try:
                import importlib.util
                spec = importlib.util.find_spec("nvidia.nccl")
                for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
                    cand = os.path.join(base, "lib", "libnccl.so.2")
                    if os.path.exists(cand):
                        os.environ["GTP_NCCL_LIB"] = cand
                        break
            except Exception:
                pass
        lib = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in _SIGS.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib
