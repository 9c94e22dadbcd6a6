"""Multi-GPU path: row-partitioned Jacobi- and AMG-PCG, one process per GPU.

Host side only does bookkeeping: the row partition, the per-rank slice of the component
table (every component that touches a row the rank owns, in global stamping order, so the
local rows of G come out bit-identical to the single-GPU assembly), the NCCL unique-id
hand-off through torch.distributed, and the call into nodal_dist_pcg (csrc/dist.cu), which
does halo discovery, halo exchange and the all-reduces natively.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .table import ComponentTable


def partition_rows(n, world):
    """Contiguous, near-equal row blocks: bounds[k] .. bounds[k+1] is rank k's range."""
    base, extra = divmod(int(n), int(world))
    sizes = np.full(world, base, dtype=np.int64)
    sizes[:extra] += 1
    bounds = np.zeros(world + 1, dtype=np.int32)
    np.cumsum(sizes, out=bounds[1:])
    return bounds


def local_component_table(table: ComponentTable, rb: int, re: int) -> ComponentTable:
    """Components with a lead on a row in [rb, re), order preserved.  Only R / A rows are
    handled (the SPD path that is partitioned); indices stay global."""
    if not table.is_spd_structured():
        raise NotImplementedError("row-partitioned solve is implemented for R / A netlists (PCG)")
    a, b = table.a, table.b
    mask = ((a >= rb) & (a < re)) | ((b >= rb) & (b < re))
    sel = np.flatnonzero(mask)
    return ComponentTable(table.type[sel], table.value[sel], a[sel], b[sel], table.c[sel], table.d[sel],
                          table.drv[sel], table.branch[sel], kcl=table.kcl, be=table.be)


def row_slice(csr, rhs, rb, re):
    """Rows [rb, re) of a CSR and rhs over all rows: (indptr rebased to 0, global indices, data, rhs slice)."""
    ip = csr.indptr[rb: re + 1]
    s, e = int(ip[0]), int(ip[-1])
    return (ip - ip[0]).contiguous(), csr.indices[s:e], csr.data[s:e], rhs[rb:re]


def broadcast_bytes(payload: bytes | None, nbytes: int, src: int = 0, device=None) -> bytes:
    """Rank `src` sends `nbytes` bytes to everyone through torch.distributed (gloo or nccl)."""
    import torch
    import torch.distributed as dist
    buf = torch.zeros(nbytes, dtype=torch.uint8)
    if dist.get_rank() == src:
        buf = torch.tensor(list(payload), dtype=torch.uint8)
    if device is not None:
        buf = buf.to(device)
    dist.broadcast(buf, src=src)
    return bytes(buf.cpu().tolist())


class DistPCG:
    """Owns the library's NCCL communicator of this rank."""

    def __init__(self, dev, rank, world):
        self.dev, self.rank, self.world = dev, int(rank), int(world)
        lib = dev.lib
        ident = None
        if self.rank == 0:
            raw = (C.c_uint8 * 128)()
            _lib.check(lib.nodal_dist_unique_id(raw), "nodal_dist_unique_id")
            ident = bytes(raw)
        if self.world > 1:
            ident = broadcast_bytes(ident, 128, src=0, device=dev.dev)
        h = C.c_void_p()
        raw = (C.c_uint8 * 128).from_buffer_copy(ident)
        _lib.check(lib.nodal_dist_create(dev.ctx, raw, self.rank, self.world, C.byref(h)), "nodal_dist_create")
        self.handle = h

    @classmethod
    def single(cls, dev):
        """One rank without a communicator (libnccl is not loaded): only solve_amg works, as the
        graph-captured single-GPU AMG-PCG."""
        self = cls.__new__(cls)
        self.dev, self.rank, self.world = dev, 0, 1
        h = C.c_void_p()
        _lib.check(dev.lib.nodal_dist_create_single(dev.ctx, C.byref(h)), "nodal_dist_create_single")
        self.handle = h
        return self

    def close(self):
        if self.handle:
            self.dev.lib.nodal_dist_destroy(self.handle)
            self.handle = None

    def assemble_local(self, table_local: ComponentTable, bounds, dtab=None):
        """Stamp + CSR build of the rank's components, then the rank's row slice.
        Returns (indptr_local, indices_global, data, rhs_local)."""
        dev = self.dev
        rb, re = int(bounds[self.rank]), int(bounds[self.rank + 1])
        csr, rhs = dev.assemble_csr(table_local, dtab=dtab)
        return row_slice(csr, rhs, rb, re)

    AMG_PARAMS = ("passes", "coarse", "omega", "scale", "maxlevels", "rounds", "direct_max", "gather_below", "max_fill")

    def solve_amg(self, n_global, bounds, indptr, indices, data, rhs_local, rtol=1e-10, maxit=None, x0=None, **params):
        """Row-partitioned AMG-preconditioned CG (csrc/dist_amg.cu)."""
        dev, torch = self.dev, self.dev.torch
        unknown = set(params) - set(self.AMG_PARAMS)
        if unknown:
            raise TypeError(f"unknown AMG parameter(s): {sorted(unknown)}")
        nloc = int(bounds[self.rank + 1] - bounds[self.rank])
        x = dev.zeros(max(2, nloc), torch.float64)[:nloc] if x0 is None else x0.clone()
        b = np.ascontiguousarray(bounds, dtype=np.int32)
        arr = (C.c_double * 9)(*[float(params.get(k, 0.0)) for k in self.AMG_PARAMS])
        iters, relres = C.c_int32(0), C.c_double(0.0)
        stats = (C.c_double * 32)()
        p = dev.ptr
        st = dev.lib.nodal_dist_amg_pcg(dev.ctx, self.handle, int(n_global), b.ctypes.data_as(C.c_void_p),
                                        int(data.numel()), p(indptr), p(indices), p(data), p(rhs_local), p(x), arr,
                                        rtol, int(maxit or 1000), C.byref(iters), C.byref(relres), stats, dev.stream())
        _lib.check(st, "nodal_dist_amg_pcg", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        nlev = int(stats[8]) + 1
        info = dict(solver="dist_amg_pcg", status=st, iterations=iters.value, relres=relres.value,
                    restarts=int(stats[2]), solve_ms=stats[3], setup_ms=stats[4], levels=int(stats[0]),
                    distributed_levels=int(stats[8]), level_rows=[int(stats[16 + l]) for l in range(min(nlev, 12))],
                    replicated_rows=int(stats[11]), coarsest_rows=int(stats[5]), coarsest_direct=bool(stats[7]),
                    comm="p2p" if stats[9] else ("nccl" if self.world > 1 else "none"),
                    kernels_per_iteration=int(stats[10]), halo_recv=int(stats[12]), nnz=int(data.numel()))
        return x, info

    def solve(self, n_global, bounds, indptr, indices, data, rhs_local, rtol=1e-10, maxit=None):
        dev, torch = self.dev, self.dev.torch
        nloc = int(bounds[self.rank + 1] - bounds[self.rank])
        x = dev.zeros(max(2, nloc), torch.float64)[:nloc]
        if maxit is None:
            maxit = max(5000, 40 * int(np.sqrt(max(n_global, 1))))
        b = np.ascontiguousarray(bounds, dtype=np.int32)
        iters, relres = C.c_int32(0), C.c_double(0.0)
        stats = (C.c_double * 16)()
        p = dev.ptr
        st = dev.lib.nodal_dist_pcg(dev.ctx, self.handle, int(n_global), b.ctypes.data_as(C.c_void_p),
                                    int(data.numel()), p(indptr), p(indices), p(data), p(rhs_local), p(x),
                                    rtol, maxit, C.byref(iters), C.byref(relres), stats, dev.stream())
        _lib.check(st, "nodal_dist_pcg", allowed=(_lib.OK, _lib.NOT_CONVERGED, _lib.BREAKDOWN))
        info = dict(solver="dist_pcg", status=st, iterations=iters.value, relres=relres.value,
                    restarts=int(stats[2]), solve_ms=stats[3], setup_ms=stats[4],
                    format="sell32" if stats[5] else "csr", stored_nnz=int(stats[6]),
                    halo_recv=int(stats[12]), halo_send=int(stats[13]), nnz=int(data.numel()),
                    comm={0: "nccl", 1: "p2p", 2: "p2p-fused"}[int(stats[9])], scaled=bool(stats[8]),
                    host_ms=dict(run=stats[14], graph_teardown=stats[15], buffer_teardown=stats[11],
                                 graph_capture=stats[10]))
        return x, info


def amg_then_jacobi(solver, rows, rhs, opts):
    """(x, info) of the row-partitioned SPD system `rows` (LocalRows) through `solver` (DistPCG): AMG-PCG
    and, when it does not converge, a Jacobi-PCG retry unless precond="amg"; Jacobi-PCG alone with
    precond="jacobi".  opts: options.SolveOptions.  A NodalLibraryError is not caught: a rank that
    fell back alone would leave the others waiting in a collective."""
    first = None
    if opts.precond != "jacobi":
        x, info = solver.solve_amg(rows.n, rows.bounds, rows.indptr, rows.indices, rows.data, rhs,
                                   rtol=opts.spd_rtol, maxit=opts.maxit, **opts.amg_params)
        if info["status"] == 0 or opts.precond == "amg":
            return x, info
        first = f"dist_amg_pcg status {info['status']}"          # same status on every rank
    x, info = solver.solve(rows.n, rows.bounds, rows.indptr, rows.indices, rows.data, rhs, rtol=opts.spd_rtol,
                           maxit=opts.maxit)
    if first:
        info["fallback_from_amg"] = first
    return x, info


class LocalRows:
    """A rank's rows of G (row pointer rebased to 0, GLOBAL column indices, device tensors)."""

    def __init__(self, n, bounds, rank, indptr, indices, data):
        self.n, self.bounds, self.rank = int(n), bounds, int(rank)
        self.indptr, self.indices, self.data = indptr, indices, data

    @property
    def nnz(self):
        return int(self.data.numel())

    @property
    def shape(self):
        return (int(self.bounds[self.rank + 1] - self.bounds[self.rank]), self.n)

    def tocsr(self):
        """Host scipy.sparse.csr_matrix of the rank's rows (container only)."""
        import scipy.sparse as sps
        return sps.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(), self.indptr.cpu().numpy()),
                              shape=self.shape)


_SOLVERS = {}


def shared_solver(dev, rank, world):
    """One NCCL communicator (and one set of peer-mapped buffers) per device and process group:
    creating them costs far more than a solve."""
    key = (dev.index, int(rank), int(world))
    if key not in _SOLVERS or not _SOLVERS[key].handle:
        _SOLVERS[key] = DistPCG(dev, rank, world)
    return _SOLVERS[key]


def single_solver(dev):
    """The communicator-free one-rank solver object of this device (graph-captured AMG-PCG)."""
    key = (dev.index, "single")
    if key not in _SOLVERS or not _SOLVERS[key].handle:
        _SOLVERS[key] = DistPCG.single(dev)
    return _SOLVERS[key]


def upload_share(dev, table, names, rank, world):
    """Rank `rank`'s contiguous 1/world share of the component table, components
    [M rank / world, M (rank + 1) / world), as device columns (the columns not in `names` are None)."""
    m = len(table)
    lo, hi = m * rank // world, m * (rank + 1) // world
    pinned = getattr(table, "_pinned", None)
    if pinned:
        share = {k: pinned[k][lo:hi].to(dev.dev, non_blocking=True) for k in names}
    else:
        share = {k: dev.to_device(getattr(table, k)[lo:hi]) for k in names}
    for k in ("type", "value", "a", "b", "c", "d", "drv", "branch"):
        share.setdefault(k, None)
    return share


def exchange_rows(dev, share, ncomp, bounds, rank, world, select):
    """The components every rank stamps, from the ranks' shares: rank s selects on the device, for every
    rank d, the components of its share that `select(columns, ncomp, rb, re)` picks for d's rows
    [bounds[d], bounds[d + 1]), and the selections travel over NVLink (torch.distributed
    all_to_all_single: plumbing).  Shares are contiguous in stamping order and are concatenated in rank
    order, so every rank receives its components in global stamping order (bit-identical rows).
    Returns (columns, count); columns that are None in `share` stay None."""
    if world == 1:
        return share, ncomp
    import torch
    import torch.distributed as dist
    names = [k for k, v in share.items() if v is not None]
    pieces, counts = [], []
    for d in range(world):
        sel, cnt = select(share, ncomp, int(bounds[d]), int(bounds[d + 1]))
        pieces.append(sel)
        counts.append(cnt)
    send_counts = torch.tensor(counts, dtype=torch.int64, device=dev.dev)
    recv_counts = torch.empty_like(send_counts)
    dist.all_to_all_single(recv_counts, send_counts)
    recv_split = [int(v) for v in recv_counts.tolist()]
    total = sum(recv_split)
    local = {k: None for k in share}
    for k in names:
        send = torch.cat([pieces[d][k][: counts[d]] for d in range(world)])
        recv = torch.empty(max(1, total), dtype=send.dtype, device=dev.dev)[:total]
        dist.all_to_all_single(recv, send, output_split_sizes=recv_split, input_split_sizes=counts)
        local[k] = recv
    return local, total


class GridRunner:
    """One rank of the row-partitioned equivalent-resistance step used by bench.py and by
    Circuit(..., distributed=True): select the rank's components ON THE DEVICE from the full
    table, stamp + build its rows, partitioned solve (Jacobi- or AMG-PCG), R on every rank."""

    def __init__(self, dev, table, probe_row, rank, world, rtol=1e-10, precond="jacobi", amg=None, solver=None):
        if not table.is_spd_structured():
            raise NotImplementedError("row-partitioned solve is implemented for R / A netlists (PCG)")
        self.dev, self.rank, self.world, self.rtol = dev, rank, world, rtol
        self.precond, self.amg = precond, dict(amg or {})
        self.table = table
        self.n = table.n
        self.bounds = partition_rows(self.n, world)
        self.probe_row = int(probe_row)
        self.owner = int(np.searchsorted(self.bounds, self.probe_row, side="right") - 1)
        self.pcg = solver if solver is not None else DistPCG(dev, rank, world)
        self._host_x = None
        self.x_local = None

    def close(self):
        self.pcg.close()

    def step_e2e(self):
        """Same step with HOST buffers: this rank's share of the component table goes up from pinned
        host memory (assemble_from_host), the rank's slice of the solution comes back to pinned
        host memory."""
        torch = self.dev.torch
        if getattr(self.table, "_pinned", None) is None:
            self.table.pin_memory()
        if self._host_x is None:
            nloc = int(self.bounds[self.rank + 1] - self.bounds[self.rank])
            self._host_x = torch.empty(nloc, dtype=torch.float64).pin_memory()
        return self.step(None, download=True)

    def assemble(self, dtab):
        """(indptr_local, indices_global, data, rhs_local) of the rank's rows from the resident table."""
        from .device import coo_stride
        dev = self.dev
        rb, re = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        ncomp = len(self.table)
        if self.world > 1:
            dtab, ncomp = dev.select_local(dtab, ncomp, rb, re)
        csr, rhs = dev.assemble_csr_raw(dtab, ncomp, self.table.kcl, self.n, coo_stride(self.table))
        return row_slice(csr, rhs, rb, re)

    def assemble_from_host(self):
        """Rows of this rank straight from the HOST table, scalable in the number of ranks: every rank
        uploads only its 1/world share of the component table (by component index), selects on the
        device which of those components touch the rows of each rank, and the selected rows travel
        over NVLink (torch.distributed all_to_all_single: plumbing) to the rank that stamps them.
        Source shares are contiguous in stamping order and are concatenated in rank order, so every
        rank sees its components in global stamping order (bit-identical rows).  Uploading the whole
        table on every rank instead costs 24 ms of host-memory bandwidth at 8 ranks."""
        from .device import coo_stride
        dev, table = self.dev, self.table
        R, r, m = self.world, self.rank, len(table)
        if not table.is_spd_structured():
            raise NotImplementedError("row-partitioned solve is implemented for R / A netlists (PCG)")
        share = upload_share(dev, table, ("type", "value", "a", "b"), r, R)
        rb, re = int(self.bounds[r]), int(self.bounds[r + 1])
        local, ncomp = exchange_rows(dev, share, m * (r + 1) // R - m * r // R, self.bounds, r, R, dev.select_local)
        csr, rhs = dev.assemble_csr_raw(local, ncomp, table.kcl, self.n, coo_stride(table))
        return row_slice(csr, rhs, rb, re)

    def step(self, dtab, download=False):
        import time
        torch = self.dev.torch
        t0 = time.perf_counter()
        indptr, indices, data, rhs = self.assemble(dtab) if dtab is not None else self.assemble_from_host()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        if self.precond == "amg":
            x, info = self.pcg.solve_amg(self.n, self.bounds, indptr, indices, data, rhs, rtol=self.rtol, **self.amg)
        else:
            x, info = self.pcg.solve(self.n, self.bounds, indptr, indices, data, rhs, rtol=self.rtol)
        t2 = time.perf_counter()
        info["assemble_wall_ms"] = (t1 - t0) * 1e3
        info["solve_wall_ms"] = (t2 - t1) * 1e3
        if download:
            self._host_x.copy_(x, non_blocking=True)
            torch.cuda.synchronize()
        r = torch.zeros(1, dtype=torch.float64, device=self.dev.dev)
        if self.rank == self.owner:
            r[0] = x[self.probe_row - int(self.bounds[self.rank])]
        nnz = torch.tensor([info["nnz"]], dtype=torch.int64, device=self.dev.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.broadcast(r, src=self.owner)
            dist.all_reduce(nnz)
        info["nnz"] = int(nnz.item())
        self.x_local = x
        return float(r.item()), info
