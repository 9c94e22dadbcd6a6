"""ctypes binding of libnodal_b200.so (the C ABI declared in include/nodal_b200.h).

There is no CPU fallback: if the shared library is missing, or no sm_100a device
is visible when a kernel is requested, the call fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnodal_b200.so")

OK, SINGULAR, NOT_CONVERGED, BREAKDOWN, CUDA_ERROR, BAD_ARG = 0, 1, 2, 3, 4, -1
PCG_FORCE_CSR, PCG_NO_GRAPH, PCG_PROFILE, PCG_NO_SCALE = 1, 2, 4, 8

_vp, _i32, _i64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double

# name -> (restype, argtypes); mirrors include/nodal_b200.h one to one
SIGNATURES = {
    "nodal_abi_version": (C.c_int, []),
    "nodal_last_error": (C.c_char_p, []),
    "nodal_launch_count": (C.c_uint64, []),
    "nodal_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "nodal_ctx_destroy": (C.c_int, [_vp]),
    "nodal_ctx_workspace_bytes": (_i64, [_vp]),
    "nodal_stamp_coo": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "nodal_csr_build": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _vp, C.POINTER(_i64), _vp]),
    "nodal_csr_build_ordered": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_csr_fetch": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp]),
    "nodal_csr_to_dense": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_coo_to_dense_atomic": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_spmv": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nodal_sell_create": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, C.POINTER(_vp), _vp]),
    "nodal_sell_destroy": (C.c_int, [_vp]),
    "nodal_sell_padded_nnz": (_i64, [_vp]),
    "nodal_sell_compact": (C.c_int, [_vp]),
    "nodal_sell_spmv": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "nodal_pcg": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _f64, _i32, _i32,
                            C.POINTER(_i32), C.POINTER(_f64), C.POINTER(_f64), _vp]),
    "nodal_gmres": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _f64, _i32, _i32,
                              C.POINTER(_i32), C.POINTER(_f64), _vp]),
    "nodal_amg_create": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, C.POINTER(_f64), C.POINTER(_vp), _vp]),
    "nodal_amg_destroy": (C.c_int, [_vp]),
    "nodal_amg_info": (C.c_int, [_vp, _i32, C.POINTER(_i32), C.POINTER(_i64), C.POINTER(_i64),
                                 C.POINTER(_f64), C.POINTER(_i32)]),
    "nodal_amg_fetch_level": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_amg_apply": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "nodal_amg_pcg": (C.c_int, [_vp, _vp, _vp, _vp, _f64, _i32, C.POINTER(_i32), C.POINTER(_f64),
                                C.POINTER(_f64), _vp]),
    "nodal_connected_components": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _vp, C.POINTER(_i32),
                                             C.POINTER(_i32), _vp]),
    "nodal_source_forest": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32] + [_vp] * 8
                            + [C.POINTER(_i64), _vp]),
    "nodal_source_reduce_scan": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, C.POINTER(_i64), _vp]),
    "nodal_source_reduce_table": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                            _vp]),
    "nodal_source_expand": (C.c_int, [_vp, _i32, _i32, _i32] + [_vp] * 9 + [_i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp,
                                                                             C.POINTER(_f64), _vp]),
    "nodal_schur_split_scan": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, C.POINTER(_i64), _vp]),
    "nodal_schur_split_place": (C.c_int, [_vp, _i32] + [_vp] * 9 + [_vp]),
    "nodal_schur_rhs_batch": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_schur_columns": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nodal_schur_branch_rhs": (C.c_int, [_vp, _i32, _i32] + [_vp] * 6 + [_vp]),
    "nodal_schur_node_rhs": (C.c_int, [_vp, _i32] + [_vp] * 6 + [_vp]),
    "nodal_schur_residual": (C.c_int, [_vp, _i32] + [_vp] * 6 + [C.POINTER(_f64), _vp]),
    "nodal_schur_add": (C.c_int, [_vp, _i64, _vp, _vp, _vp]),
    "nodal_lu_solve": (C.c_int, [_vp, _i32, _vp, _vp, _vp, C.POINTER(_i32), _vp]),
    "nodal_lu_factor": (C.c_int, [_vp, _i32, _vp, _vp, C.POINTER(_i32), _vp]),
    "nodal_lu_solve_factored": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_dgemm_sub_profile": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, C.POINTER(_f64), _vp]),
    "nodal_lu_batched": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _i32, _i32, _vp, _vp, _vp, _vp]),
    "nodal_lu_batched_soa": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _i32, _i32, _vp, _vp, _vp, _vp]),
    "nodal_dist_unique_id": (C.c_int, [_vp]),
    "nodal_dist_create": (C.c_int, [_vp, _vp, _i32, _i32, C.POINTER(_vp)]),
    "nodal_dist_create_single": (C.c_int, [_vp, C.POINTER(_vp)]),
    "nodal_dist_destroy": (C.c_int, [_vp]),
    "nodal_dist_pcg": (C.c_int, [_vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _f64, _i32,
                                 C.POINTER(_i32), C.POINTER(_f64), C.POINTER(_f64), _vp]),
    "nodal_amg_pcg_multi": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _f64, _i32, C.POINTER(_i32), C.POINTER(_f64),
                                      C.POINTER(_i32), _vp]),
    "nodal_amg_profile_sweeps": (C.c_int, [_vp, _vp, _i32, C.POINTER(_f64), _vp]),
    "nodal_amg_profile_cycle": (C.c_int, [_vp, _vp, _i32, C.POINTER(_f64), _vp]),
    "nodal_table_select_scan": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_table_select_gather": (C.c_int, [_vp, _i64, _vp, _i32, _i32] + [_vp] * 16 + [_vp]),
    "nodal_table_select_mna_scan": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, C.POINTER(_i64),
                                              _vp]),
    "nodal_table_select_mna_gather": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32] + [_vp] * 16 + [_vp]),
    "nodal_table_select_type_scan": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_table_select_type_gather": (C.c_int, [_vp, _i64, _vp, _i32] + [_vp] * 16 + [_vp]),
    "nodal_source_potentials": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nodal_source_tree_rows": (C.c_int, [_vp, _i32, _i32, _i64, _i32, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, C.POINTER(_i64), _vp]),
    "nodal_source_currents": (C.c_int, [_vp, _i32, _i32] + [_vp] * 7 + [_i32, _i64, _vp, _vp, _vp, _vp, _vp]),
    "nodal_source_residual": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, C.POINTER(_f64), _vp]),
    "nodal_source_dep_map": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_source_dep_check": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_source_dep_scan": (C.c_int, [_vp, _i32, _i32] + [_vp] * 7 + [_i32, _i32, _vp, C.POINTER(_i64), _vp]),
    "nodal_source_dep_emit": (C.c_int, [_vp, _i32, _i32] + [_vp] * 7 + [_i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "nodal_source_expand_dep": (C.c_int, [_vp, _i32, _i32, _i32] + [_vp] * 9 + [_i32, _i32, _vp, _i32, _vp, _vp, _i64,
                                                                                 _vp, _vp, _vp, _vp, C.POINTER(_f64),
                                                                                 _vp]),
    "nodal_dist_amg_pcg": (C.c_int, [_vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, C.POINTER(_f64), _f64,
                                     _i32, C.POINTER(_i32), C.POINTER(_f64), C.POINTER(_f64), _vp]),
}

_lib = None


class NodalLibraryError(RuntimeError):
    """The CUDA extension is missing or a CUDA call failed."""


def load():
    """dlopen the library and attach the prototypes (works without a GPU)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NodalLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`"
            " (or `make -C nodal_b200/csrc`). nodal_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.nodal_abi_version() != 1:
        raise NodalLibraryError("libnodal_b200.so ABI version mismatch")
    _lib = lib
    return lib


def last_error():
    return load().nodal_last_error().decode("utf-8", "replace")


def check(status, what, allowed=(OK,)):
    if status in allowed:
        return status
    raise NodalLibraryError(f"{what} failed with status {status}: {last_error()}")
