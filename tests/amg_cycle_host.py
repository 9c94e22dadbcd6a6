"""Builds (once) the CPU compilation of csrc/amg_cycle_core.cuh (tests/host_check/amg_cycle_host.cpp), the
V-cycle arithmetic the not-gpu tests run in its unfused and fused forms, and a CSR V-cycle on top of it."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def amg_cycle_host_lib():
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "host_check", "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libamg_cycle_host.so")
        src = os.path.join(HERE, "host_check", "amg_cycle_host.cpp")
        core = os.path.join(ROOT, "nodal_b200", "csrc", "amg_cycle_core.cuh")
        if (not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src),
                                                                  os.path.getmtime(core))):
            subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
        lib = C.CDLL(so)
        vp, i32, f64 = C.c_void_p, C.c_int32, C.c_double
        for name, args in (("amgc_jacobi0_host", [i32, vp, vp, f64, vp]),
                           ("amgc_prolong_host", [i32, vp, vp, f64, vp, vp]),
                           ("amgc_sweep_host", [i32, i32, vp, vp, vp, vp, vp, vp, f64, vp]),
                           ("amgc_fused_sweep_host", [i32, i32, vp, vp, vp, vp, vp, f64, vp, vp, f64, vp]),
                           ("amgc_restrict_host", [i32, vp, vp, i32, vp])):
            getattr(lib, name).restype = None
            getattr(lib, name).argtypes = args
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def cycle(M, b, fused):
    """One V(1,1) cycle of amg_mirror.AMG `M` with the kernels' arithmetic (csrc/amg.cu::cycle):
    fused=False stores x0 and the prolongated iterate, fused=True forms them where the sweeps gather.
    The coarsest level is M's (inverse or Jacobi), computed by numpy the same way in both forms."""
    lib = amg_cycle_host_lib()
    om, sc = float(M.omega), float(M.scale)
    ops = []
    for A, _, dinv, agg in M.levels:
        A = A.tocsr()
        ops.append((A.shape[0], np.ascontiguousarray(A.indptr, dtype=np.int32),
                    np.ascontiguousarray(A.indices, dtype=np.int32), np.ascontiguousarray(A.data, dtype=np.float64),
                    np.ascontiguousarray(dinv, dtype=np.float64), np.ascontiguousarray(agg, dtype=np.int32)))

    def level(l, b):
        if l == len(ops):
            return M.inv @ b if M.inv is not None else om * M.dc * b
        n, ip, ix, dv, dinv, agg = ops[l]
        nc = M.rows[l + 1]
        r = np.empty(n)
        x = np.empty(n)
        if fused:
            lib.amgc_fused_sweep_host(1, n, _p(ip), _p(ix), _p(dv), _p(dinv), _p(b), om, None, None, 0.0, _p(r))
        else:
            lib.amgc_jacobi0_host(n, _p(dinv), _p(b), om, _p(x))
            lib.amgc_sweep_host(1, n, _p(ip), _p(ix), _p(dv), _p(dinv), _p(b), _p(x), om, _p(r))
        bc = np.empty(nc)
        lib.amgc_restrict_host(n, _p(agg), _p(r), nc, _p(bc))
        xc = np.ascontiguousarray(level(l + 1, bc), dtype=np.float64)
        y = np.empty(n)
        if fused:
            lib.amgc_fused_sweep_host(2, n, _p(ip), _p(ix), _p(dv), _p(dinv), _p(b), om, _p(agg), _p(xc), sc, _p(y))
        else:
            xa = np.empty(n)
            lib.amgc_prolong_host(n, _p(agg), _p(xc), sc, _p(x), _p(xa))
            lib.amgc_sweep_host(2, n, _p(ip), _p(ix), _p(dv), _p(dinv), _p(b), _p(xa), om, _p(y))
        return y

    return level(0, np.ascontiguousarray(b, dtype=np.float64))
