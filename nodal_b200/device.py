"""Device-side plumbing: torch tensors as buffers, ctypes calls into libnodal_b200.so.

torch is used only to own device memory, streams and (in dist.py) the process
group; every kernel that runs here is one of ours.
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib
from . import constants as K
from .table import ComponentTable

_STRIDE_OF_TYPE = {K.T_R: 4, K.T_A: 2, K.T_E: 5, K.T_VCVS: 6, K.T_VCCS: 6, K.T_CCVS: 6, K.T_CCCS: 5}


def _torch():
    import torch
    return torch


def coo_stride(table: ComponentTable) -> int:
    """Slots per component the stamp kernel must reserve (see include/nodal_b200.h)."""
    need = max((_STRIDE_OF_TYPE[t] for t in table.present_types()), default=2)
    return 2 if need <= 2 else 4 if need <= 4 else need


def colbits_for(n: int) -> int:
    return max(1, int(n).bit_length())


class DeviceCSR:
    """CSR matrix + right-hand side resident in HBM (int32 indices, f64 data)."""

    def __init__(self, n, indptr, indices, data):
        self.n = int(n)
        self.indptr, self.indices, self.data = indptr, indices, data

    @property
    def nnz(self):
        return int(self.data.numel())

    @property
    def shape(self):
        return (self.n, self.n)

    def tocsr(self):
        """Host scipy.sparse.csr_matrix copy (container only -- no arithmetic)."""
        import scipy.sparse as sps
        return sps.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(),
                               self.indptr.cpu().numpy()), shape=self.shape)

    def toarray(self):
        return self.tocsr().toarray()

    def __array__(self, dtype=None, copy=None):
        a = self.toarray()
        return a if dtype is None else a.astype(dtype)


class DeviceAMG:
    """Handle of a nodal_amg hierarchy; keeps the matrix arrays alive while it exists."""

    PARAMS = ("passes", "coarse", "omega", "scale", "maxlevels", "rounds", "direct_max", "max_fill")

    def __init__(self, dev, csr, **params):
        unknown = set(params) - set(self.PARAMS)
        if unknown:
            raise TypeError(f"unknown AMG parameter(s): {sorted(unknown)}")
        self.dev, self.csr = dev, csr
        arr = (C.c_double * 8)(*[float(params.get(k, 0.0)) for k in self.PARAMS])
        h = C.c_void_p()
        p = dev.ptr
        st = dev.lib.nodal_amg_create(dev.ctx, csr.n, csr.nnz, p(csr.indptr), p(csr.indices), p(csr.data),
                                      arr, C.byref(h), dev.stream())
        _lib.check(st, "nodal_amg_create")
        self.handle = h
        cap = 64
        nl, rows, nnz = C.c_int32(0), (C.c_int64 * cap)(), (C.c_int64 * cap)()
        ms, direct = C.c_double(0.0), C.c_int32(0)
        _lib.check(dev.lib.nodal_amg_info(h, cap, C.byref(nl), rows, nnz, C.byref(ms), C.byref(direct)),
                   "nodal_amg_info")
        self.rows = [int(rows[k]) for k in range(nl.value)]
        self.nnz = [int(nnz[k]) for k in range(nl.value)]
        self.setup_ms, self.direct = ms.value, bool(direct.value)

    def close(self):
        if self.handle:
            self.dev.lib.nodal_amg_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:       # interpreter shutdown
            pass

    def aggregates(self, level):
        """Row -> aggregate map of `level` (device int32 tensor)."""
        dev = self.dev
        agg = dev.empty(max(1, self.rows[level]), dev.torch.int32)[: self.rows[level]]
        _lib.check(dev.lib.nodal_amg_fetch_level(dev.ctx, self.handle, level, dev.ptr(agg), None, None, None,
                                                 dev.stream()), "nodal_amg_fetch_level")
        return agg

    def operator(self, level):
        """The level's operator as a DeviceCSR copy."""
        dev, torch = self.dev, self.dev.torch
        n, nnz = self.rows[level], self.nnz[level]
        indptr = dev.empty(n + 1, torch.int32)
        indices = dev.empty(max(1, nnz), torch.int32)[:nnz]
        data = dev.empty(max(1, nnz), torch.float64)[:nnz]
        p = dev.ptr
        _lib.check(dev.lib.nodal_amg_fetch_level(dev.ctx, self.handle, level, None, p(indptr), p(indices),
                                                 p(data), dev.stream()), "nodal_amg_fetch_level")
        return DeviceCSR(n, indptr, indices, data)

    def apply(self, r):
        """z = M r: one V-cycle."""
        dev = self.dev
        z = dev.empty(max(1, self.csr.n), dev.torch.float64)[: self.csr.n]
        _lib.check(dev.lib.nodal_amg_apply(dev.ctx, self.handle, dev.ptr(r), dev.ptr(z), dev.stream()),
                   "nodal_amg_apply")
        return z

    def solve_multi(self, rhs, rtol=1e-10, maxit=None):
        """Several right-hand sides at once: rhs is a (K, n) device tensor, K <= 8; returns x (K, n) and
        a list of K info dicts (csrc/amg_multi.cu: every level operator is read once per sweep for all K)."""
        dev, n = self.dev, self.csr.n
        K = int(rhs.shape[0])
        if not 1 <= K <= 8 or int(rhs.shape[1]) != n:
            raise ValueError("rhs must be a (K, n) tensor with 1 <= K <= 8")
        rhs = rhs.contiguous()
        x = dev.zeros(max(2, K * n), dev.torch.float64)[: K * n].view(K, n)
        iters, relres, status = (C.c_int32 * K)(), (C.c_double * K)(), (C.c_int32 * K)()
        st = dev.lib.nodal_amg_pcg_multi(dev.ctx, self.handle, K, dev.ptr(rhs), dev.ptr(x), rtol, int(maxit or 1000),
                                         iters, relres, status, dev.stream())
        _lib.check(st, "nodal_amg_pcg_multi", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        infos = [dict(solver="amg_pcg_multi", status=int(status[k]), iterations=int(iters[k]), relres=float(relres[k]),
                      batch=K, level_rows=list(self.rows)) for k in range(K)]
        return x, infos

    def profile_sweeps(self, reps=64):
        """Average ms per launch of the level-0 SELL sweeps: dict(spmv_dot, residual, jacobi)."""
        ms = (C.c_double * 4)()
        _lib.check(self.dev.lib.nodal_amg_profile_sweeps(self.dev.ctx, self.handle, int(reps), ms, self.dev.stream()),
                   "nodal_amg_profile_sweeps")
        return dict(spmv_dot=ms[0], residual=ms[1], jacobi=ms[2])

    def profile_cycle(self, reps=64):
        """Average ms per launch of the level-0 V-cycle kernels, unfused and fused (csrc/amg.cu,
        nodal_amg_profile_cycle): dict(jacobi0, residual, prolong, jacobi, fused_residual, fused_post)."""
        ms = (C.c_double * 6)()
        _lib.check(self.dev.lib.nodal_amg_profile_cycle(self.dev.ctx, self.handle, int(reps), ms, self.dev.stream()),
                   "nodal_amg_profile_cycle")
        return dict(zip(("jacobi0", "residual", "prolong", "jacobi", "fused_residual", "fused_post"), list(ms)))

    def solve(self, rhs, rtol=1e-10, maxit=None, x0=None):
        dev, n = self.dev, self.csr.n
        x = dev.zeros(max(2, n), dev.torch.float64)[:n] if x0 is None else x0.clone()
        if maxit is None:
            maxit = 1000
        iters, relres = C.c_int32(0), C.c_double(0.0)
        stats = (C.c_double * 16)()
        st = dev.lib.nodal_amg_pcg(dev.ctx, self.handle, dev.ptr(rhs), dev.ptr(x), rtol, maxit,
                                   C.byref(iters), C.byref(relres), stats, dev.stream())
        _lib.check(st, "nodal_amg_pcg", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        info = dict(solver="amg_pcg", status=st, iterations=iters.value, relres=relres.value,
                    restarts=int(stats[2]), solve_ms=stats[3], setup_ms=stats[4], levels=int(stats[0]),
                    operator_complexity=stats[1], grid_complexity=stats[6], coarsest_rows=int(stats[5]),
                    coarsest_direct=bool(stats[7]), level_rows=list(self.rows))
        return x, info


class Device:
    """One CUDA device + one library context.  Not thread safe (one per thread)."""

    _instances = {}
    _lock = threading.Lock()

    @classmethod
    def get(cls, index=None):
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.NodalLibraryError(
                "nodal_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if index is None:
            index = torch.cuda.current_device()
        key = (threading.get_ident(), int(index))
        with cls._lock:
            if key not in cls._instances:
                cls._instances[key] = cls(int(index))
            return cls._instances[key]

    def __init__(self, index):
        self.torch = _torch()
        self.index = index
        self.dev = self.torch.device("cuda", index)
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.nodal_ctx_create(index, C.byref(h)), "nodal_ctx_create")
        self.ctx = h
        self.launches = 0   # kernels-of-ours launch counter is kept by the callers' estimates

    # ------------------------------------------------------------ helpers
    def stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)

    def empty(self, n, dtype):
        return self.torch.empty(int(n), dtype=dtype, device=self.dev)

    def zeros(self, n, dtype):
        return self.torch.zeros(int(n), dtype=dtype, device=self.dev)

    def to_device(self, arr, pin=False):
        t = self.torch.from_numpy(np.ascontiguousarray(arr))
        if pin:
            t = t.pin_memory()
        return t.to(self.dev, non_blocking=pin)

    @staticmethod
    def ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)

    def upload_table(self, table: ComponentTable, pin=False):
        """Columns of the table in HBM.  R / A-only tables (the SPD path) carry constants in the
        c / d / drv / branch columns: those are not uploaded (the kernels take null pointers for
        them), 17 instead of 33 bytes per component."""
        names = ("type", "value", "a", "b", "c", "d", "drv", "branch")
        if table.is_spd_structured():
            names = names[:4]
        if getattr(table, "_pinned", None):
            out = {name: table._pinned[name].to(self.dev, non_blocking=True) for name in names}
        else:
            out = {name: self.to_device(getattr(table, name), pin=pin) for name in names}
        for name in ("c", "d", "drv", "branch"):
            out.setdefault(name, None)
        return out

    @staticmethod
    def uploaded_bytes(table: ComponentTable):
        """Bytes upload_table moves for this table."""
        per_row = 17 if table.is_spd_structured() else 33
        return per_row * len(table)

    # ------------------------------------------------------------ stamping
    def stamp_coo(self, dtab, ncomp, kcl, n, stride):
        torch = self.torch
        cb = colbits_for(n)
        keys = self.empty(max(1, stride * ncomp), torch.int64)
        vals = self.empty(max(1, stride * ncomp), torch.float64)
        p = self.ptr
        _lib.check(self.lib.nodal_stamp_coo(
            self.ctx, ncomp, p(dtab["type"]), p(dtab["value"]), p(dtab["a"]), p(dtab["b"]),
            p(dtab["c"]), p(dtab["d"]), p(dtab["drv"]), p(dtab["branch"]),
            kcl, n, stride, cb, p(keys), p(vals), self.stream()), "nodal_stamp_coo")
        return keys, vals, cb

    def assemble_csr(self, table: ComponentTable, dtab=None, order="sorted"):
        """Stamp + CSR build.  Returns (DeviceCSR, rhs tensor).  order="first_touch" keeps the columns
        of a row in the order the reference's DOK matrix met them (what `G.tocsr()` gives before
        spsolve sorts it, nodal/nodal.py:396-397); the solvers expect the default, sorted order."""
        if dtab is None:
            dtab = self.upload_table(table)
        return self.assemble_csr_raw(dtab, len(table), table.kcl, table.n, coo_stride(table), order=order)

    def assemble_csr_raw(self, dtab, ncomp, kcl, n, stride, order="sorted"):
        """The same from device-resident columns (`dtab`: name -> tensor, `ncomp` rows used)."""
        if order not in ("sorted", "first_touch"):
            raise ValueError("order must be 'sorted' or 'first_touch'")
        keys, vals, cb = self.stamp_coo(dtab, ncomp, kcl, n, stride)
        return self._csr_from_triples(keys, vals, stride * ncomp, n, cb, 1 if order == "first_touch" else 0)

    def _csr_from_triples(self, keys, vals, nslots, n, cb, order):
        """(DeviceCSR, rhs) of `nslots` keyed triples (csrc/csr.cu: sort, in-order sums, col == n the rhs)."""
        torch = self.torch
        rhs = self.empty(max(1, n), torch.float64)[:n]
        nnz = C.c_int64(0)
        p = self.ptr
        _lib.check(self.lib.nodal_csr_build_ordered(self.ctx, n, nslots, cb, p(keys), p(vals), order, p(rhs),
                                                    C.byref(nnz), self.stream()), "nodal_csr_build")
        nnz = nnz.value
        indptr = self.empty(n + 1, torch.int32)
        indices = self.empty(max(1, nnz), torch.int32)[:nnz]
        data = self.empty(max(1, nnz), torch.float64)[:nnz]
        _lib.check(self.lib.nodal_csr_fetch(self.ctx, n, nnz, p(indptr), p(indices), p(data),
                                            self.stream()), "nodal_csr_fetch")
        # keys / vals may back the pending result until fetch has run on the stream
        self.torch.cuda.current_stream(self.dev).synchronize()
        del keys, vals
        return DeviceCSR(n, indptr, indices, data), rhs

    _COLUMNS = ("type", "value", "a", "b", "c", "d", "drv", "branch")

    def _select(self, dtab, ncomp, scan, scan_args, gather, gather_args):
        """Ordered flag / scan / gather of the rows of `dtab` that one selection of csrc/stamp.cu picks."""
        pos = self.empty(max(1, ncomp), self.torch.int32)
        count = C.c_int64(0)
        p = self.ptr
        _lib.check(getattr(self.lib, scan)(self.ctx, ncomp, *scan_args, p(pos), C.byref(count), self.stream()), scan)
        m = count.value
        out = {k: (self.empty(max(1, m), dtab[k].dtype) if dtab[k] is not None else None) for k in self._COLUMNS}
        _lib.check(getattr(self.lib, gather)(self.ctx, ncomp, p(pos), *gather_args, *[p(dtab[k]) for k in self._COLUMNS],
                                             *[p(out[k]) for k in self._COLUMNS], self.stream()), gather)
        return out, m

    def select_local(self, dtab, ncomp, rb, re):
        """Columns of the components with a lead on a row in [rb, re), order kept, selected on the
        device from the resident table (row-partitioned assembly).  Returns (columns, count)."""
        p = self.ptr
        return self._select(dtab, ncomp, "nodal_table_select_scan", (p(dtab["a"]), p(dtab["b"]), int(rb), int(re)),
                            "nodal_table_select_gather", (int(rb), int(re)))

    def select_mna_rows(self, dtab, ncomp, kcl, rb, re):
        """The same for an R / A / E table: also the E rows whose branch row kcl + branch is in [rb, re)."""
        p = self.ptr
        return self._select(dtab, ncomp, "nodal_table_select_mna_scan",
                            (p(dtab["type"]), p(dtab["a"]), p(dtab["b"]), p(dtab["branch"]), int(kcl), int(rb), int(re)),
                            "nodal_table_select_mna_gather", (int(kcl), int(rb), int(re)))

    def select_type(self, dtab, ncomp, t):
        """Columns of the components of type `t`, order kept."""
        p = self.ptr
        return self._select(dtab, ncomp, "nodal_table_select_type_scan", (p(dtab["type"]), p(dtab["a"]), p(dtab["b"]),
                                                                          int(t)),
                            "nodal_table_select_type_gather", (int(t),))

    def csr_to_dense(self, csr: DeviceCSR):
        n = csr.n
        G = self.empty(max(1, n * n), self.torch.float64)[: n * n].view(n, n)
        p = self.ptr
        _lib.check(self.lib.nodal_csr_to_dense(self.ctx, n, p(csr.indptr), p(csr.indices),
                                               p(csr.data), p(G), self.stream()), "nodal_csr_to_dense")
        return G

    def assemble_dense(self, table: ComponentTable, atomic=False):
        """Dense n x n G and rhs.  atomic=False: deterministic (sorted, in-order sums, bit-exact
        with the reference); atomic=True: warp-aggregated atomic scatter-add."""
        if not atomic:
            csr, rhs = self.assemble_csr(table)
            return self.csr_to_dense(csr), rhs
        torch = self.torch
        n, ncomp = table.n, len(table)
        stride = coo_stride(table)
        dtab = self.upload_table(table)
        keys, vals, cb = self.stamp_coo(dtab, ncomp, table.kcl, n, stride)
        G = self.empty(max(1, n * n), torch.float64)[: n * n].view(n, n)
        rhs = self.empty(max(1, n), torch.float64)[:n]
        p = self.ptr
        _lib.check(self.lib.nodal_coo_to_dense_atomic(self.ctx, n, stride * ncomp, cb, p(keys),
                                                      p(vals), p(G), p(rhs), self.stream()),
                   "nodal_coo_to_dense_atomic")
        return G, rhs

    # ------------------------------------------------------------ sparse solves
    def spmv(self, csr: DeviceCSR, x):
        y = self.empty(max(1, csr.n), self.torch.float64)[: csr.n]
        p = self.ptr
        _lib.check(self.lib.nodal_spmv(self.ctx, csr.n, csr.nnz, p(csr.indptr), p(csr.indices),
                                       p(csr.data), p(x), p(y), self.stream()), "nodal_spmv")
        return y

    def pcg(self, csr: DeviceCSR, rhs, rtol=1e-10, maxit=None, flags=0, x0=None):
        n = csr.n
        x = self.zeros(max(2, n), self.torch.float64)[:n] if x0 is None else x0.clone()
        if maxit is None:
            maxit = max(5000, 40 * int(np.sqrt(max(n, 1))))
        iters, relres = C.c_int32(0), C.c_double(0.0)
        stats = (C.c_double * 16)()
        p = self.ptr
        st = self.lib.nodal_pcg(self.ctx, n, csr.nnz, p(csr.indptr), p(csr.indices), p(csr.data),
                                p(rhs), p(x), rtol, maxit, flags, C.byref(iters), C.byref(relres),
                                stats, self.stream())
        _lib.check(st, "nodal_pcg", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        info = dict(solver="pcg", status=st, iterations=iters.value, relres=relres.value,
                    restarts=int(stats[2]), solve_ms=stats[3], setup_ms=stats[4],
                    format="sell32" if stats[5] else "csr", stored_nnz=int(stats[6]),
                    spmv_grid=int(stats[7]), scaled=bool(stats[12]))
        if stats[11]:
            info["kernel_ms"] = dict(spmv_dot=stats[8], update=stats[9], direction=stats[10],
                                     samples=int(stats[11]))
        return x, info

    def connected_components(self, table: ComponentTable, want_labels=False):
        """(number of components, nodes connected to ground, labels or None) of the lead graph:
        nodes 0..kcl-1 plus ground (= node kcl), one edge per component (csrc/graph.cu)."""
        a, b = self.to_device(table.a), self.to_device(table.b)
        labels = self.empty(table.kcl + 1, self.torch.int32) if want_labels else None
        count, reached = C.c_int32(0), C.c_int32(0)
        st = self.lib.nodal_connected_components(self.ctx, len(table), self.ptr(a), self.ptr(b), table.kcl,
                                                 self.ptr(labels) if want_labels else None,
                                                 C.byref(count), C.byref(reached), self.stream())
        _lib.check(st, "nodal_connected_components")
        return count.value, reached.value, labels

    # ------------------------------------------------------------ voltage-source elimination
    def source_forest(self, dtab, ncomp, kcl, be):
        """Forest of the E rows of a device-resident R / A / E table (csrc/sources.cu).  Returns
        (info dict, dict of device tensors); the tensors are only written when info["loops"] and
        info["branch_conflicts"] are 0."""
        torch = self.torch
        i32 = lambda k: self.empty(max(1, k), torch.int32)             # noqa: E731
        nodes = kcl + 1
        out = dict(erow=i32(be), adj_ptr=i32(nodes + 1), adj_row=i32(2 * be), rep_row=i32(nodes),
                   offset=self.empty(nodes, torch.float64), parent_edge=i32(nodes), depth=i32(nodes),
                   roots=i32(kcl))
        info = (C.c_int64 * 8)()
        p = self.ptr
        _lib.check(self.lib.nodal_source_forest(
            self.ctx, ncomp, p(dtab["type"]), p(dtab["value"]), p(dtab["a"]), p(dtab["b"]), p(dtab["branch"]),
            kcl, be, *[p(out[k]) for k in ("erow", "adj_ptr", "adj_row", "rep_row", "offset", "parent_edge",
                                           "depth", "roots")], info, self.stream()), "nodal_source_forest")
        keys = ("sources", "loops", "branch_conflicts", "trees", "floating_trees", "grounded_nodes", "rows", "depth")
        return {k: int(info[i]) for i, k in enumerate(keys)}, out

    def source_reduce(self, dtab, ncomp, kcl, forest):
        """The reduced R / A table as device columns (`dtab` form) and its number of rows."""
        torch = self.torch
        pos = self.empty(max(1, ncomp), torch.int32)
        count = C.c_int64(0)
        p = self.ptr
        args = (p(dtab["type"]), p(dtab["a"]), p(dtab["b"]), kcl, p(forest["rep_row"]), p(forest["offset"]))
        _lib.check(self.lib.nodal_source_reduce_scan(self.ctx, ncomp, *args, p(pos), C.byref(count), self.stream()),
                   "nodal_source_reduce_scan")
        m = count.value
        red = dict(type=self.empty(max(1, m), torch.uint8), value=self.empty(max(1, m), torch.float64),
                   a=self.empty(max(1, m), torch.int32), b=self.empty(max(1, m), torch.int32),
                   c=None, d=None, drv=None, branch=None)
        _lib.check(self.lib.nodal_source_reduce_table(
            self.ctx, ncomp, p(dtab["type"]), p(dtab["value"]), p(dtab["a"]), p(dtab["b"]), kcl,
            p(forest["rep_row"]), p(forest["offset"]), p(pos), p(red["type"]), p(red["value"]), p(red["a"]),
            p(red["b"]), self.stream()), "nodal_source_reduce_table")
        return red, m

    def source_expand(self, dtab, kcl, forest, info, y, csr: DeviceCSR, rhs):
        """x = [potentials; source currents] of the full system from the reduced solution y, and
        ||rhs - G x|| / ||rhs|| with the full MNA matrix `csr`."""
        n = csr.n
        x = self.empty(max(1, n), self.torch.float64)[:n]
        relres = C.c_double(0.0)
        p = self.ptr
        f = forest
        _lib.check(self.lib.nodal_source_expand(
            self.ctx, kcl, n, info["sources"], p(f["erow"]), p(dtab["a"]), p(dtab["b"]), p(dtab["branch"]),
            p(f["adj_ptr"]), p(f["adj_row"]), p(f["rep_row"]), p(f["offset"]), p(f["depth"]), info["depth"],
            p(y), p(rhs), csr.nnz, p(csr.indptr), p(csr.indices), p(csr.data), p(x), C.byref(relres),
            self.stream()), "nodal_source_expand")
        return x, relres.value

    # the stages of source_expand for a rank's rows of the full MNA matrix (dist_sources.py)
    def source_potentials(self, kcl, n, forest, y):
        """x (n): the potentials of every node from the reduced solution y, 0 on the branch rows."""
        x = self.empty(max(1, n), self.torch.float64)[:n]
        p = self.ptr
        _lib.check(self.lib.nodal_source_potentials(self.ctx, kcl, n, p(forest["rep_row"]), p(forest["offset"]), p(y),
                                                    p(x), self.stream()), "nodal_source_potentials")
        return x

    def source_tree_rows(self, kcl, n, nnz_full, rb, re, forest, rows, rhs, x):
        """(row, rhs, G x) of the rows in [rb, re) whose node hangs in a source tree (depth >= 1), in row
        order; `rows` is the rank's LocalRows of the full matrix (n rows, nnz_full entries in all)."""
        torch = self.torch
        cap = max(1, re - rb)
        row, o_rhs, o_gx = self.empty(cap, torch.int32), self.empty(cap, torch.float64), self.empty(cap, torch.float64)
        count = C.c_int64(0)
        p = self.ptr
        _lib.check(self.lib.nodal_source_tree_rows(
            self.ctx, kcl, n, nnz_full, rb, re, p(forest["depth"]), p(rhs), rows.nnz, p(rows.indptr), p(rows.indices),
            p(rows.data), p(x), p(row), p(o_rhs), p(o_gx), C.byref(count), self.stream()), "nodal_source_tree_rows")
        k = count.value
        return row[:k], o_rhs[:k], o_gx[:k]

    def source_currents(self, kcl, etab, forest, info, tree_row, tree_rhs, tree_gx, x):
        """Source currents into x[kcl + branch] from the tree rows of all ranks (E-only table `etab`)."""
        p, f = self.ptr, forest
        _lib.check(self.lib.nodal_source_currents(
            self.ctx, kcl, info["sources"], p(f["erow"]), p(etab["a"]), p(etab["b"]), p(etab["branch"]),
            p(f["adj_ptr"]), p(f["adj_row"]), p(f["depth"]), info["depth"], int(tree_row.numel()), p(tree_row),
            p(tree_rhs), p(tree_gx), p(x), self.stream()), "nodal_source_currents")

    def source_residual(self, n, nnz_full, rows, rhs, x):
        """(sum (rhs - G x)^2, sum rhs^2) over the rank's rows (LocalRows of the full matrix)."""
        sums = (C.c_double * 2)()
        p = self.ptr
        _lib.check(self.lib.nodal_source_residual(self.ctx, n, nnz_full, int(rhs.numel()), p(rhs), rows.nnz,
                                                  p(rows.indptr), p(rows.indices), p(rows.data), p(x), sums,
                                                  self.stream()), "nodal_source_residual")
        return sums[0], sums[1]

    # ------------------------------------------------------------ E rows plus dependent branch rows
    def source_dep_map(self, dtab, ncomp, be):
        """(d_map, dependent branches, branches not owned by exactly one component): d_map (be) numbers
        the dependent branches in branch order, -1 for the others."""
        d_map = self.empty(max(1, be), self.torch.int32)
        info = (C.c_int64 * 2)()
        _lib.check(self.lib.nodal_source_dep_map(self.ctx, ncomp, self.ptr(dtab["type"]), self.ptr(dtab["branch"]), be,
                                                 self.ptr(d_map), info, self.stream()), "nodal_source_dep_map")
        return d_map, int(info[0]), int(info[1])

    def source_dep_check(self, dtab, ncomp, kcl, forest):
        """Number of VCVS / VCCS / CCVS rows whose output leads lie in one source tree."""
        count = C.c_int64(0)
        p = self.ptr
        _lib.check(self.lib.nodal_source_dep_check(self.ctx, ncomp, p(dtab["type"]), p(dtab["a"]), p(dtab["b"]), kcl,
                                                   p(forest["rep_row"]), C.byref(count), self.stream()),
                   "nodal_source_dep_check")
        return count.value

    def source_dep_assemble(self, red, nred, mn, md, kcl, forest, d_map, G: DeviceCSR, rhs):
        """(DeviceCSR, rhs) of the reduced system (mn + md rows, sorted columns): the triples of the
        reduced R / A table's stamp, then those of nodal_source_dep_emit, summed in that order."""
        torch = self.torch
        nr = mn + md
        cb = colbits_for(nr)
        p = self.ptr
        pos = self.empty(max(1, G.n), torch.int32)
        cnt = C.c_int64(0)
        args = (p(G.indptr), p(G.indices), p(G.data), p(rhs), p(forest["rep_row"]), p(forest["offset"]), p(d_map),
                mn, nr)
        _lib.check(self.lib.nodal_source_dep_scan(self.ctx, G.n, kcl, *args, p(pos), C.byref(cnt), self.stream()),
                   "nodal_source_dep_scan")
        ns, nd = 4 * nred, cnt.value                     # stride of R rows (A rows need 2)
        keys = self.empty(max(1, ns + nd), torch.int64)
        vals = self.empty(max(1, ns + nd), torch.float64)
        if nred > 0:
            _lib.check(self.lib.nodal_stamp_coo(self.ctx, nred, p(red["type"]), p(red["value"]), p(red["a"]),
                                                p(red["b"]), None, None, None, None, mn, nr, 4, cb, p(keys), p(vals),
                                                self.stream()), "nodal_stamp_coo")
        _lib.check(self.lib.nodal_source_dep_emit(self.ctx, G.n, kcl, *args, cb, p(pos), p(keys[ns:]), p(vals[ns:]),
                                                  self.stream()), "nodal_source_dep_emit")
        return self._csr_from_triples(keys, vals, ns + nd, nr, cb, 0)

    def source_expand_dep(self, etab, kcl, forest, info, d_map, mn, y, csr: DeviceCSR, rhs):
        """source_expand on a table with dependent branch rows: `etab` the E-only table the forest was
        built on (with the table's branch numbers), y = [reduced node rows; dependent currents]."""
        n = csr.n
        x = self.empty(max(1, n), self.torch.float64)[:n]
        relres = C.c_double(0.0)
        p, f = self.ptr, forest
        _lib.check(self.lib.nodal_source_expand_dep(
            self.ctx, kcl, n, info["sources"], p(f["erow"]), p(etab["a"]), p(etab["b"]), p(etab["branch"]),
            p(f["adj_ptr"]), p(f["adj_row"]), p(f["rep_row"]), p(f["offset"]), p(f["depth"]), info["depth"], n - kcl,
            p(d_map), mn, p(y), p(rhs), csr.nnz, p(csr.indptr), p(csr.indices), p(csr.data), p(x), C.byref(relres),
            self.stream()), "nodal_source_expand_dep")
        return x, relres.value

    # ------------------------------------------------------------ Schur complement of the branch rows
    def schur_split(self, G: DeviceCSR, kcl):
        """(L, B) of the sorted MNA matrix G (csrc/schur.cu): L the DeviceCSR of the node-node block,
        B a dict of device tensors ptr (kcl + 1), col (branch index), val: the node rows' branch entries."""
        torch = self.torch
        p = self.ptr
        l_ptr, b_ptr = self.empty(kcl + 1, torch.int32), self.empty(kcl + 1, torch.int32)
        nnz = (C.c_int64 * 2)()
        _lib.check(self.lib.nodal_schur_split_scan(self.ctx, kcl, p(G.indptr), p(G.indices), p(l_ptr), p(b_ptr), nnz,
                                                   self.stream()), "nodal_schur_split_scan")
        nl, nb = int(nnz[0]), int(nnz[1])
        l_idx, l_val = self.empty(max(1, nl), torch.int32)[:nl], self.empty(max(1, nl), torch.float64)[:nl]
        b_col, b_val = self.empty(max(1, nb), torch.int32)[:nb], self.empty(max(1, nb), torch.float64)[:nb]
        _lib.check(self.lib.nodal_schur_split_place(self.ctx, kcl, p(G.indptr), p(G.indices), p(G.data), p(l_ptr),
                                                    p(l_idx), p(l_val), p(b_ptr), p(b_col), p(b_val), self.stream()),
                   "nodal_schur_split_place")
        return DeviceCSR(kcl, l_ptr, l_idx, l_val), dict(ptr=b_ptr, col=b_col, val=b_val)

    def schur_rhs_batch(self, kcl, j0, K, B):
        """(K, kcl) device tensor: the branch columns j0 .. j0 + K - 1 of B."""
        rhs = self.empty(max(2, K * kcl), self.torch.float64)[: K * kcl].view(K, kcl)
        p = self.ptr
        _lib.check(self.lib.nodal_schur_rhs_batch(self.ctx, kcl, j0, K, p(B["ptr"]), p(B["col"]), p(B["val"]), p(rhs),
                                                  self.stream()), "nodal_schur_rhs_batch")
        return rhs

    def schur_columns(self, G: DeviceCSR, kcl, j0, Z, S):
        """S[:, j0 : j0 + K] = D - C Z (S: the m x m device tensor, Z: (K, kcl))."""
        m, K = int(S.shape[0]), int(Z.shape[0])
        p = self.ptr
        _lib.check(self.lib.nodal_schur_columns(self.ctx, kcl, m, j0, K, p(G.indptr), p(G.indices), p(G.data),
                                                p(Z.contiguous()), p(S), self.stream()), "nodal_schur_columns")

    def schur_branch_rhs(self, G: DeviceCSR, kcl, r, t):
        """r[kcl:] - C t (m entries)."""
        m = G.n - kcl
        out = self.empty(max(1, m), self.torch.float64)[:m]
        p = self.ptr
        _lib.check(self.lib.nodal_schur_branch_rhs(self.ctx, kcl, m, p(G.indptr), p(G.indices), p(G.data), p(r), p(t),
                                                   p(out), self.stream()), "nodal_schur_branch_rhs")
        return out

    def schur_node_rhs(self, kcl, B, r, xb):
        """r[:kcl] - B xb (kcl entries)."""
        out = self.empty(max(1, kcl), self.torch.float64)[:kcl]
        p = self.ptr
        _lib.check(self.lib.nodal_schur_node_rhs(self.ctx, kcl, p(B["ptr"]), p(B["col"]), p(B["val"]), p(r), p(xb),
                                                 p(out), self.stream()), "nodal_schur_node_rhs")
        return out

    def schur_residual(self, G: DeviceCSR, rhs, x, r):
        """r = rhs - G x in place; returns (sum r^2, sum rhs^2)."""
        sums = (C.c_double * 2)()
        p = self.ptr
        _lib.check(self.lib.nodal_schur_residual(self.ctx, G.n, p(G.indptr), p(G.indices), p(G.data), p(rhs), p(x),
                                                 p(r), sums, self.stream()), "nodal_schur_residual")
        return sums[0], sums[1]

    def schur_add(self, x, d):
        """x += d (same length)."""
        _lib.check(self.lib.nodal_schur_add(self.ctx, int(d.numel()), self.ptr(x), self.ptr(d), self.stream()),
                   "nodal_schur_add")

    def r_grounded(self, dtab, ncomp, kcl):
        """True when every node reaches ground through the R rows of the device table alone."""
        rt, nr = self.select_type(dtab, ncomp, K.T_R)
        count, reached = C.c_int32(0), C.c_int32(0)
        _lib.check(self.lib.nodal_connected_components(self.ctx, nr, self.ptr(rt["a"]), self.ptr(rt["b"]), kcl, None,
                                                       C.byref(count), C.byref(reached), self.stream()),
                   "nodal_connected_components")
        return reached.value == kcl + 1

    def amg(self, csr: DeviceCSR, **params):
        """Aggregation-AMG hierarchy for an SPD DeviceCSR (csrc/amg.cu); see DeviceAMG."""
        return DeviceAMG(self, csr, **params)

    def amg_pcg(self, csr: DeviceCSR, rhs, rtol=1e-10, maxit=None, x0=None, **params):
        """AMG-preconditioned CG, hierarchy built and dropped inside the call."""
        amg = DeviceAMG(self, csr, **params)
        try:
            return amg.solve(rhs, rtol=rtol, maxit=maxit, x0=x0)
        finally:
            amg.close()

    def gmres(self, csr: DeviceCSR, rhs, rtol=1e-12, restart=60, maxit=20000):
        n = csr.n
        x = self.zeros(max(2, n), self.torch.float64)[:n]
        iters, relres = C.c_int32(0), C.c_double(0.0)
        p = self.ptr
        st = self.lib.nodal_gmres(self.ctx, n, csr.nnz, p(csr.indptr), p(csr.indices), p(csr.data),
                                  p(rhs), p(x), rtol, restart, maxit, C.byref(iters),
                                  C.byref(relres), self.stream())
        _lib.check(st, "nodal_gmres", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        return x, dict(solver="gmres", status=st, iterations=iters.value, relres=relres.value)

    # ------------------------------------------------------------ dense solves
    def lu_solve(self, G, rhs):
        """Solves G x = rhs; G (n x n, row-major) is overwritten by its LU factors."""
        n = int(G.shape[0])
        x = self.empty(max(1, n), self.torch.float64)[:n]
        info = C.c_int32(0)
        p = self.ptr
        st = self.lib.nodal_lu_solve(self.ctx, n, p(G), p(rhs), p(x), C.byref(info), self.stream())
        _lib.check(st, "nodal_lu_solve", allowed=(_lib.OK, _lib.SINGULAR))
        return x, dict(solver="lu", status=st, info=info.value)

    def lu_factor(self, G):
        """P G = L U in place (G: n x n row-major device tensor); returns (ipiv, info dict)."""
        n = int(G.shape[0])
        ipiv = self.empty(max(1, n), self.torch.int32)[:n]
        info = C.c_int32(0)
        st = self.lib.nodal_lu_factor(self.ctx, n, self.ptr(G), self.ptr(ipiv), C.byref(info), self.stream())
        _lib.check(st, "nodal_lu_factor", allowed=(_lib.OK, _lib.SINGULAR))
        return ipiv, dict(solver="lu", status=st, info=info.value)

    def lu_solve_factored(self, LU, ipiv, rhs):
        """x for one rhs with the factors of lu_factor."""
        n = int(LU.shape[0])
        x = self.empty(max(1, n), self.torch.float64)[:n]
        p = self.ptr
        _lib.check(self.lib.nodal_lu_solve_factored(self.ctx, n, p(LU), p(ipiv), p(rhs), p(x), self.stream()),
                   "nodal_lu_solve_factored")
        return x

    def lu_batched(self, table: ComponentTable, values, layout="aos"):
        """Batched small-system solve.  layout "aos": values (batch, ncomp) -> x (batch, n);
        layout "soa": values (ncomp, batch) -> x (n, batch), the coalesced form (n <= 8).
        Returns x, info (batch,)."""
        torch = self.torch
        if layout not in ("aos", "soa"):
            raise ValueError("layout must be 'aos' or 'soa'")
        soa = layout == "soa"
        batch, ncomp = (int(values.shape[1]), int(values.shape[0])) if soa else (int(values.shape[0]), int(values.shape[1]))
        if ncomp != len(table):
            raise ValueError("values must have one entry per component of the topology")
        if not values.is_contiguous():
            values = values.contiguous()
        n = table.n
        dtab = self.upload_table(table)
        x = self.empty(max(1, batch * n), torch.float64)[: batch * n]
        x = x.view(n, batch) if soa else x.view(batch, n)
        info = self.empty(max(1, batch), torch.int32)[:batch]
        p = self.ptr
        fn = self.lib.nodal_lu_batched_soa if soa else self.lib.nodal_lu_batched
        _lib.check(fn(self.ctx, batch, ncomp, p(dtab["type"]), p(dtab["a"]), p(dtab["b"]), p(dtab["c"]),
                      p(dtab["d"]), p(dtab["drv"]), p(dtab["branch"]), table.kcl, n, p(values), p(x),
                      p(info), self.stream()), "nodal_lu_batched")
        return x, info
