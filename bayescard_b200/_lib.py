"""ctypes binding of ``libbayescard_b200.so`` (the C ABI declared in ``include/bayescard_b200.h``).

No torch types cross this boundary: callers pass raw addresses (``tensor.data_ptr()``,
``ndarray.ctypes.data``) and a raw ``cudaStream_t``.  There is no fallback of any kind: if the
shared library is missing, :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbayescard_b200.so")
SPEC_CACHE_DIR = os.path.join(_HERE, "_spec_cache")

BC_OK = 0
DESC_RANGE_U8, DESC_RANGE_U16, DESC_DENSE_F32, DESC_BITS = 0, 1, 2, 3
ELIMIT = -5
SQLC_BITS, SQLC_DENSE, SQLC_ZERO, SQLC_PYTHON, SQLC_OVERFLOW = 0, 1, 2, 3, 4
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_SPEC, KERNEL_GEMM, KERNEL_GEMM_SIMT, KERNEL_FUSED = 0, 1, 2, 3, 4, 5

_lib = None


class BayesCardError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile the extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    script = os.path.join(_HERE, "csrc", "build.sh")
    res = subprocess.run(["bash", script], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise BayesCardError("building libbayescard_b200.so failed")
    global _lib
    _lib = None
    return LIB_PATH


_SIGS = {
    # name: (restype, argtypes)
    "bc_model_create": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "bc_model_create_from_file": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "bc_model_destroy": (None, [C.c_void_p]),
    "bc_model_n_nodes": (C.c_int, [C.c_void_p]),
    "bc_model_device": (C.c_int, [C.c_void_p]),
    "bc_model_dense_width": (C.c_int64, [C.c_void_p]),
    "bc_model_dense_offset": (C.c_int64, [C.c_void_p, C.c_int]),
    "bc_model_bits_offset": (C.c_int64, [C.c_void_p, C.c_int]),
    "bc_model_bits_default": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "bc_model_desc_stride": (C.c_int64, [C.c_void_p, C.c_int]),
    "bc_model_flops_dense": (C.c_int64, [C.c_void_p]),
    "bc_model_specialize": (C.c_int, [C.c_void_p, C.c_char_p]),
    "bc_model_has_spec": (C.c_int, [C.c_void_p]),
    "bc_model_fused_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "bc_model_fused_sequence": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int32)]),
    "bc_model_spec_source": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "bc_model_spec_hash": (C.c_uint64, [C.c_void_p]),
    "bc_model_load_cubin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "bc_model_specialize_marginal": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p]),
    "bc_model_marginal_source": (C.c_int64, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "bc_model_marginal_hash": (C.c_uint64, [C.c_void_p, C.c_int]),
    "bc_marginal_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "bc_expectation_marginal_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                                C.c_void_p]),
    "bc_joint_marginal_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                          C.c_int, C.c_void_p]),
    "bc_model_specialize_joint": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "bc_model_joint_source": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "bc_model_joint_hash": (C.c_uint64, [C.c_void_p, C.c_int, C.c_int]),
    "bc_query_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_void_p]),
    "bc_query_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "bc_query_batch_scaled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p]),
    "bc_query_batch_scaled_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "bc_convert_desc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]),
    "bc_expand_sparse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "bc_query_batch_sparse_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                             C.c_int]),
    "bc_model_packed_geometry": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "bc_pack_sparse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                 C.POINTER(C.c_size_t)]),
    "bc_expand_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "bc_query_batch_packed_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                             C.c_void_p, C.c_int]),
    "bc_query_batch_packed_host_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                                    C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "bc_pipe_wait": (C.c_int, [C.c_void_p, C.c_uint64]),
    "bc_expand_wsparse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "bc_query_batch_wsparse_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                              C.c_int]),
    "bc_gen_sparse_queries_host": (C.c_int, [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]),
    "bc_gen_range_queries": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p]),
    "bc_gen_range_queries_host": (C.c_int, [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_int,
                                            C.c_int, C.c_void_p]),
    "bc_sqlc_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "bc_sqlc_destroy": (None, [C.c_void_p]),
    "bc_sqlc_set_null": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "bc_sqlc_column_index": (C.c_int, [C.c_void_p, C.c_char_p]),
    "bc_sqlc_compile_factors": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t),
                                          C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "bc_joblight_create": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_double, C.POINTER(C.c_void_p)]),
    "bc_joblight_destroy": (None, [C.c_void_p]),
    "bc_joblight_plan": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "bc_joblight_plan_text": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "bc_joblight_combine": (C.c_int, [C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bc_sqlc_bits_stride": (C.c_int64, [C.c_void_p]),
    "bc_sqlc_dense_width": (C.c_int64, [C.c_void_p]),
    "bc_sqlc_add_categorical": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "bc_sqlc_add_continuous": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "bc_sqlc_compile": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                  C.c_void_p, C.POINTER(C.c_size_t)]),
    "bc_fit_counts": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t,
                                C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.c_void_p]),
    "bc_model_set_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "bc_model_get_counts": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bc_model_arena": (C.c_int64, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "bc_model_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_size_t, C.c_void_p,
                                  C.POINTER(C.c_uint32), C.c_void_p]),
    "bc_pair_counts": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p,
                                 C.c_size_t, C.POINTER(C.c_uint32), C.c_void_p]),
    "bc_chow_liu": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p,
                              C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]),
    "bc_measure_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "bc_launch_count": (C.c_uint64, []),
    "bc_last_error": (C.c_char_p, []),
    "bc_version": (C.c_char_p, []),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib():
    """The loaded library.  Raises if the CUDA extension has not been built -- no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BayesCardError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(bayescard_b200 has no CPU fallback)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc: int) -> None:
    if rc != BC_OK:
        raise BayesCardError(f"bayescard_b200 error {rc}: {lib().bc_last_error().decode('utf-8', 'replace')}")
