"""ctypes binding of libbicgstab_b200.so (include/bicgstab_b200.h).

The shared library is the product; this module only declares its C ABI to Python.  There is no Python or
CPU fallback: if the library has not been built the import fails, and the compute entry points themselves
exit(1) when no Blackwell GPU is usable (reference error convention, solver.c:43-46).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbicgstab_b200.so")


class CSR_Matrix(C.Structure):
    """matrix.h:19-26 -- double *val; unsigned *col; unsigned *ptr; unsigned nz, rows, cols."""
    _fields_ = [("val", C.POINTER(C.c_double)), ("col", C.POINTER(C.c_uint)), ("ptr", C.POINTER(C.c_uint)),
                ("nz", C.c_uint), ("rows", C.c_uint), ("cols", C.c_uint)]


class INFO_Matrix(C.Structure):
    """matrix.h:28-33 -- unsigned nz, rows, cols; MM_typecode code; int *recvcounts; int *displs."""
    _fields_ = [("nz", C.c_uint), ("rows", C.c_uint), ("cols", C.c_uint), ("code", C.c_char * 4),
                ("recvcounts", C.POINTER(C.c_int)), ("displs", C.POINTER(C.c_int))]


class bicg_stats(C.Structure):
    _fields_ = [("iters", C.c_int), ("converged", C.c_int), ("final_res", C.c_double), ("loop_ms", C.c_double),
                ("h2d_ms", C.c_double), ("d2h_ms", C.c_double), ("upload_ms", C.c_double),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("kernel_launches", C.c_int),
                ("spmv_lanes", C.c_int), ("spmv_kind", C.c_int)]


ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)

# every symbol include/bicgstab_b200.h declares: (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    # Part 1 -- the reference's interface
    "csr_init_matrix": (None, [_P(CSR_Matrix)]),
    "csr_free_matrix": (None, [_P(CSR_Matrix)]),
    "csr_shift_diagonal": (None, [_P(CSR_Matrix), C.c_double]),
    "MPI_csr_load_matrix_block": (None, [C.c_char_p, _P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix)]),
    "MPI_csr_spmv_ovlap": (None, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p, C.c_void_p]),
    "bicgstab": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p]),
    "ca_bicgstab": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p]),
    "pipe_bicgstab": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p]),
    "pipe_bicgstab_rr": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "shifted_lopbicg_switching": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "shifted_lopbicg_switching_noovlp": (C.c_int, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    # vector.h:4-7 on host arrays (csrc/hostvec.cpp): what the shifted drivers prepare their right-hand sides with
    "my_daxpy": (None, [C.c_int, C.c_double, _P(C.c_double), _P(C.c_double)]),
    "my_ddot": (C.c_double, [C.c_int, _P(C.c_double), _P(C.c_double)]),
    "my_dscal": (None, [C.c_int, C.c_double, _P(C.c_double)]),
    "my_dcopy": (None, [C.c_int, _P(C.c_double), _P(C.c_double)]),
    # Part 2 -- extensions
    "bicg_abi_version": (C.c_int, []),
    "bicg_set_option": (C.c_int, [C.c_char_p, C.c_char_p]),
    "bicg_comm_init": (C.c_int, [C.c_int, C.c_int, ALLGATHER_FN, C.c_void_p]),
    "bicg_comm_finalize": (None, []),
    "bicg_comm_rank": (C.c_int, []),
    "bicg_comm_world": (C.c_int, []),
    "bicg_matrix_create": (C.c_void_p, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix)]),
    "bicg_matrix_destroy": (None, [C.c_void_p]),
    "bicg_matrix_invalidate": (None, [_P(CSR_Matrix)]),
    "bicg_solve": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, _P(bicg_stats)]),
    "bicg_shifted_solve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, _P(bicg_stats)]),
    "bicg_last_shift_info": (C.c_int, [_P(C.c_int), _P(C.c_int), C.c_int]),
    "bicg_spmv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bicg_spmv_time": (C.c_int, [C.c_void_p, C.c_int, _P(C.c_double), _P(C.c_double)]),
    "bicg_profile_solve": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _P(C.c_double), _P(C.c_int)]),
    "bicg_debug_vec_phase": (C.c_int, [C.c_void_p, C.c_int, _P(C.c_double), C.c_void_p, _P(C.c_double)]),
    "bicg_debug_spmv_epi": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, _P(C.c_double)]),
    "bicg_debug_get_vec": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "bicg_debug_get_scalars": (C.c_int, [C.c_void_p, _P(C.c_double)]),
    "bicg_debug_resident_ctas": (C.c_int, [C.c_void_p]),
    "bicg_debug_mega_tiles": (C.c_int, [C.c_void_p, _P(C.c_int)]),
    "bicg_last_history": (C.c_int, [_P(C.c_double), C.c_int]),
    "bicg_last_stats": (_P(bicg_stats), []),
    "bicg_stream": (C.c_void_p, []),
    "bicg_device": (C.c_int, []),
    "bicg_synchronize": (None, []),
    "bicg_host_alloc": (C.c_void_p, [C.c_size_t]),
    "bicg_host_free": (None, [C.c_void_p]),
    "bicg_plan_partition": (None, [C.c_int, C.c_int, _P(C.c_int), _P(C.c_int)]),
    "bicg_plan_partition_nnz": (None, [_P(C.c_uint), C.c_int, C.c_int, _P(C.c_int), _P(C.c_int)]),
    "bicg_plan_tiles": (C.c_int, [_P(C.c_uint), C.c_int, C.c_int, C.c_int, _P(C.c_int), C.c_int]),
    "bicg_plan_cta_tiles": (C.c_int, [_P(C.c_uint), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, _P(C.c_int), C.c_int,
                                      _P(C.c_int), _P(C.c_uint)]),
    "bicg_plan_cta_tiles_capped": (C.c_int, [_P(C.c_uint), C.c_int, C.c_int, C.c_int, C.c_int, _P(C.c_int), _P(C.c_uint), _P(C.c_int),
                                             C.c_int, _P(C.c_int), _P(C.c_uint)]),
    "bicg_plan_halo_runs": (C.c_int, [_P(CSR_Matrix), _P(INFO_Matrix), C.c_int, C.c_int, C.c_int, _P(C.c_int), C.c_int]),
    "bicg_plan_merge": (C.c_longlong, [_P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix), C.c_int, C.c_int, C.c_int, C.c_int,
                                       _P(C.c_uint), _P(C.c_uint), _P(C.c_double), _P(C.c_int), C.c_int, _P(C.c_int)]),
    "bicg_comm_selftest": (C.c_int, []),
    "bicg_plan_push_runs": (C.c_int, [_P(C.c_int), _P(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, _P(C.c_int), C.c_int]),
    "bicg_gen_block": (C.c_int, [C.c_int, C.c_longlong, C.c_double, C.c_uint64, C.c_int, C.c_int,
                                 _P(CSR_Matrix), _P(CSR_Matrix), _P(INFO_Matrix)]),
    "bicg_shm_bootstrap": (C.c_int, []),
    "bicg_shm_shutdown": (None, []),
}


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C mpi-bicgstab_b200/csrc`). There is no Python/CPU fallback.")
    lib = C.CDLL(LIB_PATH)          # RTLD_LOCAL: our bicgstab()/... must not interpose on other libraries
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here = the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()
