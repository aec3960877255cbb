"""ctypes binding of the C ABI in include/sqpb200.h (libsqpb200.so).

The library is the product: if it is missing or cannot be loaded this module raises; there is no
Python / CPU fallback for any numerical entry point.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SQPB200_LIB") or os.path.join(HERE, "lib", "libsqpb200.so")

LOC_HOST, LOC_DEVICE = 0, 1
LP, QP = 1, 2
VEC_G, VEC_LB, VEC_UB, VEC_LBA, VEC_UBA = 0, 1, 2, 3, 4
MAT_A, MAT_H = 0, 1
QP_OPTIMAL = 20

#: every symbol include/sqpb200.h declares (tests check that the .so exports all of them)
EXPORTS = [
    "sqpb200_default_options", "sqpb200_version", "sqpb200_device_count", "sqpb200_create", "sqpb200_destroy",
    "sqpb200_set_stream", "sqpb200_synchronize", "sqpb200_last_error", "sqpb200_set_structure_A",
    "sqpb200_set_structure_H", "sqpb200_set_structure_csc", "sqpb200_get_structure", "sqpb200_get_nnz",
    "sqpb200_set_values_A", "sqpb200_set_values_H", "sqpb200_set_values_csc", "sqpb200_get_values_csc",
    "sqpb200_set_vectors", "sqpb200_get_vectors", "sqpb200_qphandler_bounds", "sqpb200_qphandler_g",
    "sqpb200_solve", "sqpb200_get_solution", "sqpb200_get_working_set", "sqpb200_kkt_residuals",
    "sqpb200_kkt_residuals_recompute", "sqpb200_spmv", "sqpb200_assemble_csc_batched", "sqpb200_launch_count",
    "sqpb200_solve_config", "sqpb200_last_solve_ms", "sqpb200_get_profile", "sqpb200_io_layout", "sqpb200_solve_host", "sqpb200_vector_reduce", "sqpb200_vector_elementwise",
    "sqpb200_nlp_compile", "sqpb200_nlp_cubin_size", "sqpb200_nlp_load", "sqpb200_nlp_eval", "sqpb200_nlp_destroy",
    "sqpb200_nlp_launch_count", "sqpb200_nlp_last_error",
    "sqpb200_sqp_phase", "sqpb200_sqp_optimize", "sqpb200_sqp_optimize_stream", "sqpb200_reset", "sqpb200_solve_device_mask", "sqpb200_device_buffers", "sqpb200_solve_per_instance",
    "sqpb200_sqp_graph_create", "sqpb200_sqp_graph_launch", "sqpb200_sqp_graph_destroy",
    # QORE layout: compressed-row matrices, stacked bounds / primal / dual / working set
    "sqpb200_set_structure_A_csr", "sqpb200_set_structure_H_csr", "sqpb200_set_structure_csr", "sqpb200_get_structure_csr",
    "sqpb200_set_values_csr", "sqpb200_get_values_csr", "sqpb200_set_bounds_stacked", "sqpb200_get_bounds_stacked",
    "sqpb200_get_solution_stacked",
]


class Options(C.Structure):
    _fields_ = [("qp_maxiter", C.c_int), ("lp_maxiter", C.c_int), ("enable_flipping", C.c_int),
                ("enable_ramping", C.c_int), ("enable_drift", C.c_int), ("team_size", C.c_int),
                ("keep_state", C.c_int), ("factor_cap", C.c_int), ("debug_force_error_branch", C.c_int),
                ("refactorise_every", C.c_int)]


_LIB = None


def lib():
    """Load libsqpb200.so (raises if it has not been built: see restartsqp_b200.build)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libsqpb200.so is missing (%s): run `python -m restartsqp_b200.build`; "
                               "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.sqpb200_version.restype = C.c_char_p
        L.sqpb200_last_error.restype = C.c_char_p
        L.sqpb200_last_error.argtypes = [C.c_void_p]
        L.sqpb200_launch_count.restype = C.c_longlong
        L.sqpb200_launch_count.argtypes = [C.c_void_p]
        L.sqpb200_get_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.sqpb200_io_layout.argtypes = [C.c_void_p] * 5
        L.sqpb200_reset.argtypes = [C.c_void_p]
        L.sqpb200_set_structure_A_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 4
        L.sqpb200_set_structure_H_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.sqpb200_set_structure_csr.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.sqpb200_get_structure_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqpb200_set_values_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.sqpb200_get_values_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.sqpb200_set_bounds_stacked.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.sqpb200_get_bounds_stacked.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sqpb200_get_solution_stacked.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sqpb200_vector_reduce.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.sqpb200_vector_elementwise.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]
        L.sqpb200_sqp_optimize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p]
        L.sqpb200_sqp_optimize_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqpb200_sqp_graph_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
        L.sqpb200_sqp_graph_launch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqpb200_sqp_graph_destroy.argtypes = [C.c_void_p]
        L.sqpb200_solve_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqpb200_last_solve_ms.restype = C.c_float
        L.sqpb200_last_solve_ms.argtypes = [C.c_void_p]
        L.sqpb200_nlp_last_error.restype = C.c_char_p
        L.sqpb200_nlp_cubin_size.restype = C.c_longlong
        L.sqpb200_nlp_cubin_size.argtypes = [C.c_void_p]
        L.sqpb200_nlp_launch_count.restype = C.c_longlong
        L.sqpb200_nlp_launch_count.argtypes = [C.c_void_p]
        L.sqpb200_nlp_compile.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_void_p]
        L.sqpb200_nlp_load.argtypes = [C.c_void_p, C.c_int]
        L.sqpb200_nlp_destroy.argtypes = [C.c_void_p]
        L.sqpb200_nlp_eval.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p]
        _LIB = L
    return _LIB


class SqpB200Error(RuntimeError):
    pass


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def ptr(a):
    """(void*, loc) for a numpy array (host) or a torch tensor (host or CUDA)."""
    if a is None:
        return None, LOC_HOST
    if _is_torch(a):
        assert a.is_contiguous()
        return C.c_void_p(a.data_ptr()), (LOC_DEVICE if a.is_cuda else LOC_HOST)
    assert isinstance(a, np.ndarray) and a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data), LOC_HOST


def f64(a):
    if _is_torch(a):
        import torch
        assert a.dtype == torch.float64
        return a.contiguous()
    return np.ascontiguousarray(a, dtype=np.float64)


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)
