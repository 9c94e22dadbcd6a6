"""Builds (once) the CPU compilation of csrc/schur_core.cuh (tests/host_check/schur_host.cpp), the
Schur-complement rules the not-gpu tests check against schur_mirror.py."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def schur_host_lib():
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "host_check", "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libschur_host.so")
        src = os.path.join(HERE, "host_check", "schur_host.cpp")
        core = os.path.join(ROOT, "nodal_b200", "csrc", "schur_core.cuh")
        if (not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src),
                                                                  os.path.getmtime(core))):
            subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
        lib = C.CDLL(so)
        vp, i32 = C.c_void_p, C.c_int32
        for name, args in (("schur_counts_host", [i32] + [vp] * 4),
                           ("schur_columns_host", [i32] * 4 + [vp] * 5),
                           ("schur_branch_rhs_host", [i32, i32] + [vp] * 6),
                           ("schur_node_rhs_host", [i32] + [vp] * 6),
                           ("schur_residual_host", [i32] + [vp] * 6)):
            fn = getattr(lib, name)
            fn.restype = None
            fn.argtypes = args
        _lib = lib
    return _lib
