"""Builds (once) the CPU compilation of csrc/sources_core.cuh (tests/host_check/sources_host.cpp), the
voltage-source elimination rules the not-gpu tests check against sources_mirror.py."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def sources_host_lib():
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "host_check", "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libsources_host.so")
        src = os.path.join(HERE, "host_check", "sources_host.cpp")
        core = os.path.join(ROOT, "nodal_b200", "csrc", "sources_core.cuh")
        if (not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src),
                                                                  os.path.getmtime(core))):
            subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
        lib = C.CDLL(so)
        lib.src_offsets_host.restype = None
        lib.src_offsets_host.argtypes = [C.c_int32] + [C.c_void_p] * 5 + [C.c_int32, C.c_void_p]
        lib.src_reduce_table_host.restype = C.c_int64
        lib.src_reduce_table_host.argtypes = [C.c_int64] + [C.c_void_p] * 4 + [C.c_int32] + [C.c_void_p] * 6
        lib.src_expand_host.restype = None
        lib.src_expand_host.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32] + [C.c_void_p] * 6
        _lib = lib
    return _lib
