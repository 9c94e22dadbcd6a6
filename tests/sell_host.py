"""Builds (once) the CPU compilation of csrc/sell_core.cuh (tests/host_check/sell_host.cpp): the per-entry
rules of the SELL entry encodings, and a host SELL-32 fill in both encodings on top of them."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def sell_host_lib():
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "host_check", "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libsell_host.so")
        src = os.path.join(HERE, "host_check", "sell_host.cpp")
        core = os.path.join(ROOT, "nodal_b200", "csrc", "sell_core.cuh")
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(core)):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
        lib = C.CDLL(so)
        vp, i32 = C.c_void_p, C.c_int32
        lib.sellh_plan.restype = C.c_int
        lib.sellh_plan.argtypes = [i32, vp, vp, vp, vp, vp, vp]
        lib.sellh_fill.restype = None
        lib.sellh_fill.argtypes = [i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
        lib.sellh_decode.restype = None
        lib.sellh_decode.argtypes = [i32, vp, vp, vp, vp, vp, vp]
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def build(n, indptr, indices, data):
    """SELL-32 of a CSR matrix in both encodings: dict(compact, fits, ndict, dict, slice_w, cols, vals,
    dcol, vidx, dcols, dvals), the last two the compact entries decoded (None when wide)."""
    lib = sell_host_lib()
    indptr = np.ascontiguousarray(indptr, dtype=np.int32)
    indices = np.ascontiguousarray(indices, dtype=np.int32)
    data = np.ascontiguousarray(data, dtype=np.float64)
    fits, ndict = C.c_int32(0), C.c_int32(0)
    dct = np.zeros(256, dtype=np.uint64)
    compact = bool(lib.sellh_plan(n, _p(indptr), _p(indices), _p(data), C.byref(fits), _p(dct), C.byref(ndict)))
    ns = (n + 31) // 32
    lens = np.zeros(ns * 32, dtype=np.int64)
    lens[:n] = np.diff(indptr)
    widths = lens.reshape(ns, 32).max(axis=1) if ns else np.zeros(0, dtype=np.int64)
    slice_w = np.concatenate([[0], np.cumsum(widths)]).astype(np.uint32)
    padded = int(slice_w[-1]) * 32
    cols = np.zeros(padded, dtype=np.int32)
    vals = np.zeros(padded, dtype=np.float64)
    dcol = np.zeros(padded, dtype=np.int16)
    vidx = np.zeros(padded, dtype=np.uint8)
    lib.sellh_fill(n, _p(indptr), _p(indices), _p(data), _p(slice_w), _p(dct) if compact else None, ndict.value,
                   _p(cols), _p(vals), _p(dcol), _p(vidx))
    out = dict(compact=compact, fits=bool(fits.value), ndict=ndict.value, dict=dct[: ndict.value], slice_w=slice_w,
               cols=cols, vals=vals, dcol=dcol, vidx=vidx, dcols=None, dvals=None)
    if compact:
        out["dcols"] = np.zeros(padded, dtype=np.int32)
        out["dvals"] = np.zeros(padded, dtype=np.float64)
        lib.sellh_decode(n, _p(slice_w), _p(dcol), _p(vidx), _p(dct), _p(out["dcols"]), _p(out["dvals"]))
    return out
