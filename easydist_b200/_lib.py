"""ctypes binding of libedb.so — the C-ABI declared in include/edb.h.

This is the reference-side binding a maintainer would add (see INTEGRATION.md): the reference's
reshard ops are Python callables (easydist/torch/passes/sharding.py:94-168), so the FFI is ctypes.
The product path fails loudly when the library is missing: there is no CPU fallback.
"""
import ctypes
import os
from ctypes import (POINTER, c_char_p, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p)

from . import build as _build

EDB_OK, EDB_E_INVALID, EDB_E_UNSUPPORTED, EDB_E_CUDA, EDB_E_STATE = 0, 1, 2, 3, 4

DTYPE_CODES = {"float32": 0, "bfloat16": 1, "float16": 2, "float64": 3, "int32": 4, "int64": 5}
REDOP_CODES = {"sum": 0, "max": 1, "min": 2, "avg": 3}


class EdbError(RuntimeError):
    """A libedb call failed (mirrors the reference raising RuntimeError/AssertionError)."""

    def __init__(self, code, msg):
        super().__init__(f"libedb error {code}: {msg}")
        self.code = code


class EdbUnsupported(EdbError):
    """The kernel does not cover this shape/layout; the dispatcher may route elsewhere."""


_I64P = POINTER(c_int64)
_IP = POINTER(c_int)

# name -> (restype, argtypes); every symbol include/edb.h declares
SIGNATURES = {
    "edb_version": (c_int, []),
    "edb_last_error": (c_char_p, []),
    "edb_init": (c_int, [c_int, c_int, c_int, c_size_t]),
    "edb_finalize": (c_int, []),
    "edb_is_initialized": (c_int, []),
    "edb_health": (c_int, []),
    "edb_heap_info": (c_int, [POINTER(c_void_p), POINTER(c_size_t), POINTER(c_size_t)]),
    "edb_ipc_export": (c_int, [c_void_p]),
    "edb_ipc_attach": (c_int, [c_int, c_void_p]),
    "edb_attach_local": (c_int, [c_int, c_void_p]),
    "edb_group_create": (c_int, [_IP, c_int, c_int, _IP]),
    "edb_group_info": (c_int, [c_int, _IP, _IP]),
    "edb_symm_alloc": (c_int, [c_size_t, c_size_t, POINTER(c_uint64)]),
    "edb_symm_mark": (c_int, [POINTER(c_uint64)]),
    "edb_symm_reset": (c_int, [c_uint64]),
    "edb_scatter": (c_int, [c_void_p, c_void_p, _I64P, c_int, c_int, c_int, c_int, c_int, _I64P,
                            c_void_p]),
    "edb_copy": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "edb_box_copy_local": (c_int, [c_void_p, _I64P, c_void_p, _I64P, _I64P, c_int, c_int,
                                   c_void_p]),
    "edb_all_gather": (c_int, [c_int, c_uint64, c_void_p, _I64P, c_int, c_int, c_int, c_void_p]),
    "edb_reduce_scatter": (c_int, [c_int, c_void_p, c_uint64, c_void_p, _I64P, c_int, c_int, c_int,
                                   c_int, c_float, c_int, c_void_p]),
    "edb_all_reduce": (c_int, [c_int, c_void_p, c_uint64, c_uint64, c_void_p, c_int64, c_int, c_int,
                               c_void_p]),
    "edb_all_to_all": (c_int, [c_int, c_void_p, c_uint64, c_void_p, _I64P, c_int, c_int, c_int,
                               c_int, c_void_p]),
    "edb_box_exchange": (c_int, [c_int, c_void_p, _I64P, c_uint64, c_void_p, _I64P, c_int, c_int,
                                 c_int, _IP, _I64P, _I64P, _I64P, _I64P, c_void_p]),
    "edb_halo_exchange": (c_int, [c_int, c_void_p, c_uint64, c_void_p, _I64P, c_int, c_int, c_int,
                                  c_int, c_void_p]),
    "edb_gemm_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                              c_int64, c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "edb_epoch_barrier": (c_int, [c_int, c_void_p]),
    "edb_all_gather_push": (c_int, [c_int, c_uint64, c_void_p, _I64P, c_int, c_int, c_int, c_void_p]),
    "edb_all_to_all_push": (c_int, [c_int, c_uint64, c_void_p, _I64P, c_int, c_int, c_int, c_int,
                                    c_void_p]),
    "edb_reduce_scatter_push": (c_int, [c_int, c_void_p, c_uint64, c_void_p, _I64P, c_int, c_int,
                                        c_int, c_int, c_float, c_int, c_void_p]),
    "edb_all_reduce_push": (c_int, [c_int, c_uint64, c_uint64, c_void_p, c_int64, c_int, c_int,
                                    c_void_p]),
    "edb_ag_gemm_epoch_bf16": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_uint64, c_uint64,
                                       c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "edb_ag_prefetch": (c_int, [c_int, c_int, c_void_p, c_void_p, _I64P, _I64P, _I64P, c_void_p]),
    "edb_gemm_pf_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                 c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p,
                                 c_void_p, _I64P, _I64P, _I64P, c_void_p]),
    "edb_gemm_epi_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                                  c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_int,
                                  c_int, c_int, c_void_p, c_void_p, _I64P, _I64P, _I64P, c_void_p]),
    "edb_gemm_push_bf16": (c_int, [c_int, c_uint64, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                   c_int64, c_int64, c_int, c_int, c_void_p]),
    "edb_rs_finish_local": (c_int, [c_int, c_int, c_void_p, c_void_p, _I64P, c_float, c_int,
                                    c_void_p]),
    "edb_layer_norm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int64, c_int64, c_float, c_int, c_void_p]),
    "edb_layer_norm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p]),
    "edb_layer_norm_bwd_add": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                       c_int, c_void_p]),
    "edb_layer_norm_bwd_workspace": (c_int, [c_int64, POINTER(c_size_t)]),
    "edb_colsum": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "edb_colsum_workspace": (c_int, [c_int64, POINTER(c_size_t)]),
    "edb_cross_entropy_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                      c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "edb_cross_entropy_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int,
                                      c_void_p]),
    "edb_sgd_momentum": (c_int, [c_int, c_void_p, c_void_p, c_void_p, _I64P, c_float, c_float, c_float,
                                 c_int, c_void_p]),
    "edb_set_option": (c_int, [c_char_p, c_int64]),
    "edb_get_option": (c_int, [c_char_p, POINTER(c_int64)]),
    "edb_launch_count": (c_uint64, []),
}

_lib = None


def lib_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load libedb.so (building it first when sources are newer and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if build_if_missing and _build._nvcc() is not None and _build.needs_build():
        _build.build()
    if not os.path.exists(path):
        raise EdbError(EDB_E_STATE,
                       f"{path} is missing and cannot be built here (no nvcc); run "
                       "`python -m easydist_b200.build` where nvcc is available")
    lib = ctypes.CDLL(path, mode=ctypes.RTLD_GLOBAL)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # raises AttributeError if the header and the .so drift apart
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc == EDB_OK:
        return
    msg = load().edb_last_error().decode("utf-8", "replace")
    if rc == EDB_E_UNSUPPORTED:
        raise EdbUnsupported(rc, msg)
    raise EdbError(rc, msg)


def i64_array(values):
    values = [int(v) for v in values]
    return (c_int64 * max(1, len(values)))(*values)


def int_array(values):
    values = [int(v) for v in values]
    return (c_int * max(1, len(values)))(*values)
