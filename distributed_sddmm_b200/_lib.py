"""ctypes binding of include/hnh_b200.h (the C ABI of libhnh_b200.so)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class LibraryMissing(RuntimeError):
    pass


def library_path() -> str:
    return os.path.join(_HERE, "libhnh_b200.so")


# name -> (restype, argtypes); every symbol declared in include/hnh_b200.h
_P = C.c_void_p
_I64 = C.c_int64
ABI = {
    "hnh_abi_version": (C.c_int, []),
    "hnh_build_info": (C.c_char_p, []),
    "hnh_last_error_string": (C.c_char_p, []),
    "hnh_launch_count": (C.c_uint64, []),
    "hnh_sddmm_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, C.c_int, C.c_int, _P]),
    "hnh_sddmm_scaled_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "hnh_sddmm_coo_f64": (C.c_int, [_P, _P, _P, _I64, _P, _P, C.c_int, C.c_int, _P]),
    "hnh_spmm_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, C.c_int, C.c_int, _P]),
    "hnh_fused_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, _P, C.c_int, C.c_int, _P]),
    "hnh_fused_scaled_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "hnh_fill_f64": (C.c_int, [_P, _I64, C.c_double, _P]),
    "hnh_random_uniform_f64": (C.c_int, [_P, _I64, C.c_uint64, _P]),
    "hnh_hadamard_f64": (C.c_int, [_P, _P, _P, _I64, _P]),
    "hnh_expand_row_idx": (C.c_int, [_P, _I64, _I64, _P, _P]),
    "hnh_batch_dot_f64": (C.c_int, [_P, _P, _P, _I64, C.c_int, _P]),
    "hnh_row_axpy_f64": (C.c_int, [_P, _P, C.c_double, _P, _P, _I64, C.c_int, _P]),
    "hnh_vec_quotient_f64": (C.c_int, [_P, _P, C.c_double, _P, C.c_double, _I64, _P]),
    "hnh_axpby_f64": (C.c_int, [_P, C.c_double, _P, C.c_double, _P, _I64, _P]),
    "hnh_squared_norm_f64": (C.c_int, [_P, _P, _I64, _P]),
    "hnh_leaky_relu_f64": (C.c_int, [_P, _P, _I64, C.c_double, _P]),
    "hnh_relu_cols_f64": (C.c_int, [_P, _I64, _I64, _P, _I64, _I64, _P]),
    "hnh_dgemm_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _P]),
    "hnh_relu_cols_backward_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _P]),
    "hnh_leaky_relu_slope_f64": (C.c_int, [_P, _P, _I64, C.c_double, _P]),
    "hnh_dgemm_tn_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _P]),
    "hnh_dgemm_nt_f64": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, C.c_double, _P]),
    "hnh_block_create_host": (C.c_int, [_P, _P, _I64, _I64, _I64, C.c_int, C.POINTER(_P)]),
    "hnh_block_destroy": (None, [_P]),
    "hnh_block_run_host": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_int, C.c_int, _P]),
    "hnh_er_generate_host": (C.c_int64, [C.c_int, C.c_int, C.c_uint64, _I64, _I64, _P, _P, _P, _I64]),
    "hnh_coo_to_csr_host": (C.c_int, [_I64, _I64, _I64, _P, _P, _P, C.c_int, _P, _P, _P, _P]),
    "hnh_sddmm_coo_host": (C.c_int, [_P, _P, _P, _I64, _P, _I64, _P, _I64, C.c_int]),
    "hnh_spmm_host": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _I64, _P, C.c_int]),
    "hnh_er_generate_device": (C.c_int64, [C.c_int, C.c_int, C.c_uint64, _I64, _I64, _P, _P, _P, _I64, _P]),
    "hnh_coo_to_csr_device": (C.c_int, [_I64, _I64, _I64, _P, _P, _P, C.c_int, _P, _P, _P, _P, _P]),
    "hnh_tuples_bucket_by_owner_device": (C.c_int, [_P, _P, _P, _I64, C.c_int, _I64, _I64, _P, _I64, _I64, C.c_int, _P, _P, _P, _P, _P]),
    "hnh_tuples_sort_colmajor_device": (C.c_int, [_P, _P, _P, _I64, C.c_uint64, C.c_uint64, _P]),
    "hnh_tuples_mod_device": (C.c_int, [_P, _P, _I64, C.c_uint64, C.c_uint64, _P]),
    "hnh_tuples_block_starts_device": (C.c_int, [_P, _I64, C.c_uint64, C.c_int, _P, _P]),
}


def _preload_bundled_nccl():
    """libhnh_b200.so needs `libnccl.so.2`.  When PyTorch shares the process it brings its own, newer
    NCCL under the same soname; whichever copy is mapped first serves both.  Map PyTorch's copy first
    (when there is one) so that a later `import torch` still finds every symbol it was built against."""
    import sys
    for base in sys.path:
        cand = os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
            except OSError:
                pass
            return


def lib():
    """Load libhnh_b200.so (built in-tree by build.py).  Raises LibraryMissing loudly when it
    has not been built -- the product has no fallback path."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise LibraryMissing(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`"
                " (nvcc, sm_100a).  distributed_sddmm_b200 has no CPU fallback.")
        _preload_bundled_nccl()
        L = C.CDLL(path)
        for name, (res, args) in ABI.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc: int, what: str = "hnh call") -> None:
    if rc != 0:
        msg = lib().hnh_last_error_string().decode()
        raise RuntimeError(f"{what} failed with code {rc}: {msg}")


# ---- driver ABI (include/hnh_b200_driver.h) --------------------------------------------------
class AlgDims(C.Structure):
    _fields_ = [("M", C.c_int64), ("N", C.c_int64), ("R", C.c_int64), ("p", C.c_int), ("c", C.c_int),
                ("localArows", C.c_int), ("localAcols", C.c_int), ("localBrows", C.c_int),
                ("localBcols", C.c_int), ("s_values", C.c_int64), ("st_values", C.c_int64),
                ("r_split", C.c_int), ("grid_i", C.c_int), ("grid_j", C.c_int), ("grid_k", C.c_int),
                ("n_a_submatrices", C.c_int), ("n_b_submatrices", C.c_int)]


_SZ = C.c_size_t
_PSZ = C.POINTER(C.c_size_t)
CB_SENDRECV = C.CFUNCTYPE(C.c_int, _P, C.c_int, _P, _SZ, C.c_int, _P, _SZ, C.c_int)
CB_ALLGATHER = C.CFUNCTYPE(C.c_int, _P, C.c_int, _P, _P, _SZ)
CB_REDUCE_SCATTER = C.CFUNCTYPE(C.c_int, _P, C.c_int, _P, _P, _SZ)
CB_ALLREDUCE = C.CFUNCTYPE(C.c_int, _P, C.c_int, _P, _SZ)
CB_ALLTOALLV = C.CFUNCTYPE(C.c_int, _P, C.c_int, _P, _PSZ, _PSZ, _P, _PSZ, _PSZ)
CB_BARRIER = C.CFUNCTYPE(C.c_int, _P, C.c_int)
CB_SPLIT = C.CFUNCTYPE(C.c_int, _P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                       C.POINTER(C.c_int))


class ExternalTransport(C.Structure):
    _fields_ = [("ctx", _P), ("sendrecv", CB_SENDRECV), ("allgather", CB_ALLGATHER),
                ("reduce_scatter_f64", CB_REDUCE_SCATTER), ("allreduce_f64", CB_ALLREDUCE),
                ("alltoallv", CB_ALLTOALLV), ("barrier", CB_BARRIER), ("split", CB_SPLIT)]


_PP = C.POINTER(_P)
ABI.update({
    "hnhd_init_self": (C.c_int, []),
    "hnhd_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "hnhd_init_nccl": (C.c_int, [C.c_int, C.c_int, C.c_char_p]),
    "hnhd_init_external": (C.c_int, [C.c_int, C.c_int, C.POINTER(ExternalTransport)]),
    "hnhd_finalize": (C.c_int, []),
    "hnhd_world_rank": (C.c_int, []),
    "hnhd_world_size": (C.c_int, []),
    "hnhd_barrier": (C.c_int, []),
    "hnhd_device_synchronize": (C.c_int, []),
    "hnhd_spmat_load_er": (C.c_int, [C.c_int, C.c_int, C.c_uint64, _PP]),
    "hnhd_spmat_load_file": (C.c_int, [C.c_char_p, _PP]),
    "hnhd_spmat_from_tuples": (C.c_int, [C.c_uint64, C.c_uint64, _P, _P, _P, _I64, _PP]),
    "hnhd_spmat_info": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                  C.POINTER(C.c_int64)]),
    "hnhd_spmat_tuples": (C.c_int, [_P, _P, _P, _P, _I64]),
    "hnhd_spmat_destroy": (None, [_P]),
    "hnhd_alg_create": (C.c_int, [C.c_char_p, _P, C.c_int, C.c_int, _PP]),
    "hnhd_alg_destroy": (None, [_P]),
    "hnhd_alg_dims": (C.c_int, [_P, C.POINTER(AlgDims)]),
    "hnhd_alg_submatrices": (C.c_int, [_P, C.c_int, _P, C.c_int]),
    "hnhd_setup_times_json": (C.c_int, [C.c_char_p, _SZ, C.c_int]),
    "hnhd_alg_info_json": (C.c_int, [_P, C.c_char_p, _SZ]),
    "hnhd_alg_perf_json": (C.c_int, [_P, C.c_char_p, _SZ]),
    "hnhd_alg_reset_timers": (C.c_int, [_P]),
    "hnhd_alg_block_count": (C.c_int, [_P, C.c_int]),
    "hnhd_alg_block_meta": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hnhd_alg_block_arrays": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "hnhd_dense_create": (C.c_int, [_I64, _I64, C.c_double, _PP]),
    "hnhd_dense_like": (C.c_int, [_P, C.c_int, C.c_double, _PP]),
    "hnhd_dense_fill": (C.c_int, [_P, C.c_double]),
    "hnhd_dense_dummy_initialize": (C.c_int, [_P, _P, C.c_int]),
    "hnhd_dense_from_host": (C.c_int, [_P, _P]),
    "hnhd_dense_to_host": (C.c_int, [_P, _P]),
    "hnhd_dense_shape": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hnhd_dense_data": (_P, [_P]),
    "hnhd_dense_destroy": (None, [_P]),
    "hnhd_vec_create": (C.c_int, [_I64, C.c_double, _PP]),
    "hnhd_vec_like": (C.c_int, [_P, C.c_int, C.c_double, _PP]),
    "hnhd_vec_fill": (C.c_int, [_P, C.c_double]),
    "hnhd_vec_from_host": (C.c_int, [_P, _P]),
    "hnhd_vec_to_host": (C.c_int, [_P, _P]),
    "hnhd_vec_size": (C.c_int64, [_P]),
    "hnhd_vec_destroy": (None, [_P]),
    "hnhd_alg_op": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_int]),
    "hnhd_alg_fused_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int64]),
    "hnhd_als_run": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "hnhd_gat_create": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int), C.c_double, _PP]),
    "hnhd_gat_weight_shape": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hnhd_gat_set_weight": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "hnhd_gat_buffer_shape": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hnhd_gat_set_input": (C.c_int, [_P, _P]),
    "hnhd_gat_get_buffer": (C.c_int, [_P, C.c_int, _P]),
    "hnhd_gat_forward": (C.c_int, [_P]),
    "hnhd_gat_supports_backward": (C.c_int, [_P]),
    "hnhd_gat_backward": (C.c_int, [_P, _P]),
    "hnhd_gat_get_weight_grad": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "hnhd_gat_get_input_grad": (C.c_int, [_P, _P]),
    "hnhd_gat_get_weight": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "hnhd_gat_sgd_step": (C.c_int, [_P, C.c_double]),
    "hnhd_gat_destroy": (None, [_P]),
    "hnhd_timer_start": (C.c_int, []),
    "hnhd_timer_stop": (C.c_int, [C.POINTER(C.c_double)]),
    "hnhd_als_residuals": (C.c_int, [_P, C.c_int, _P]),
    "hnhd_benchmark_algorithm": (C.c_int, [_P, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                           C.c_int, C.c_int, C.c_char_p, _SZ]),
})
