"""Builds (once) the CPU compilation of the dependent-row rules of csrc/sources_core.cuh
(tests/host_check/source_schur_host.cpp), checked by the not-gpu tests against source_schur_mirror.py."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def source_schur_host_lib():
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "host_check", "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libsource_schur_host.so")
        src = os.path.join(HERE, "host_check", "source_schur_host.cpp")
        deps = [src] + [os.path.join(ROOT, "nodal_b200", "csrc", h) for h in ("sources_core.cuh", "schur_core.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
        lib = C.CDLL(so)
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        lib.source_dep_triples_host.restype = i64
        lib.source_dep_triples_host.argtypes = [i32, i32] + [vp] * 7 + [i32, i32] + [vp] * 3
        lib.source_dep_collapsed_host.restype = i64
        lib.source_dep_collapsed_host.argtypes = [i64, vp, vp, vp, i32, vp]
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def dep_triples(indptr, indices, data, rhs, kcl, f, d_map, mn, nr):
    """(rows, cols, vals) of src_dep_row over every row of the full sorted CSR."""
    lib = source_schur_host_lib()
    indptr = np.ascontiguousarray(indptr, np.int32)
    indices = np.ascontiguousarray(indices, np.int32)
    data, rhs = np.ascontiguousarray(data, np.float64), np.ascontiguousarray(rhs, np.float64)
    rep = np.ascontiguousarray(f["rep_row"], np.int32)
    off = np.ascontiguousarray(f["offset"], np.float64)
    d_map = np.ascontiguousarray(d_map, np.int32)
    n = len(indptr) - 1
    args = (n, kcl, _p(indptr), _p(indices), _p(data), _p(rhs), _p(rep), _p(off), _p(d_map), mn, nr)
    cnt = lib.source_dep_triples_host(*args, None, None, None)
    rows, cols, vals = np.empty(cnt, np.int64), np.empty(cnt, np.int64), np.empty(cnt, np.float64)
    assert lib.source_dep_triples_host(*args, _p(rows), _p(cols), _p(vals)) == cnt
    return rows, cols, vals


def collapsed(table, f):
    lib = source_schur_host_lib()
    rep = np.ascontiguousarray(f["rep_row"], np.int32)
    return lib.source_dep_collapsed_host(len(table), _p(table.type), _p(table.a), _p(table.b), table.kcl, _p(rep))
