"""Row-partitioned solve of R / A / E netlists through the elimination of the voltage sources:
Circuit(netlist, sparse=True, distributed=True) under torchrun, one process per GPU, for netlists whose
E rows form a forest (sources.py gives the single-GPU form; tests/test_dist_sources_host.py states
this one in numpy).

Rank r of R uploads only its share of the table, components [M r / R, M (r + 1) / R), and only the
columns R / A / E stamping and the forest read (type, value, a, b, branch: csrc/stamp_core.cuh).
  build   the rank's rows [rb, re) of the full MNA matrix over partition_rows(n, R): every share
          selects, per destination rank, the components that write its rows (a lead in the range, or
          an E row whose branch row is), the selections are exchanged (dist.exchange_rows), stamped
          and built; the rows are bit-identical to the single-GPU assembly of the whole table.
  forest  the E rows of every share, compacted in order and all-gathered in rank order: every rank
          holds the E-only table in global order and runs the unchanged forest on it (replicated).
  reduce  every rank reduces its own share with that forest (the rule is per component, so the
          shares' reduced tables concatenated in rank order are the single-GPU reduced table), the
          reduced rows are exchanged over partition_rows(m, R), built, and solved with the
          row-partitioned AMG-PCG (Jacobi-PCG retry unless precond="amg").
  expand  y all-gathered; every rank forms all potentials; each rank forms G x on its rows of the
          full matrix and contributes (row, rhs, G x) of its rows that hang in a source tree; with
          those all-gathered every rank runs the subtree sums and holds every source current,
          bit-identical to the single-GPU expansion of the same y.  relres_full adds the ranks' sums
          of squares on the host in rank order (deterministic for a given world size).
"""
from __future__ import annotations

import time

import numpy as np

from . import constants as K
from . import dist as ndist
from . import sources

# what R / A / E stamping and the forest read; c / d / drv only matter for dependent sources
_COLUMNS = ("type", "value", "a", "b", "branch")


def _allgather(dev, cols, count, world):
    """Every rank's `count` rows of the device columns `cols`, concatenated in rank order.
    Returns (columns, total, counts of the ranks); None columns stay None."""
    if world == 1:
        return cols, count, [count]
    import torch
    import torch.distributed as dist
    torch_dev = dev.dev
    mine = torch.tensor([count], dtype=torch.int64, device=torch_dev)
    counts = torch.empty(world, dtype=torch.int64, device=torch_dev)
    dist.all_gather_into_tensor(counts, mine)
    counts = [int(v) for v in counts.tolist()]
    pad, total = max(1, max(counts)), sum(counts)
    out = {}
    for k, v in cols.items():
        if v is None:
            out[k] = None
            continue
        send = torch.zeros(pad, dtype=v.dtype, device=torch_dev)
        send[:count] = v[:count]
        recv = torch.empty(world * pad, dtype=v.dtype, device=torch_dev)
        dist.all_gather_into_tensor(recv, send)
        out[k] = torch.cat([recv[d * pad: d * pad + counts[d]] for d in range(world)])
    return out, total, counts


def _rows_of(dev, csr, rhs, bounds, rank):
    """The rank's rows [rb, re) of a CSR built over all rows: (LocalRows, rhs slice)."""
    indptr, indices, data, rhs = ndist.row_slice(csr, rhs, int(bounds[rank]), int(bounds[rank + 1]))
    return ndist.LocalRows(csr.n, bounds, rank, indptr, indices, data), rhs


class DistSources:
    """One rank of the row-partitioned eliminated solve of a Circuit (see the module docstring)."""

    def __init__(self, circuit, dev, table, rank, world):
        from .device import coo_stride
        # one rule at any size: there is no other row-partitioned path for E rows
        reason = sources.skip_reason(table, True, 0)
        if circuit.opts.eliminate_sources is False:
            raise NotImplementedError("row-partitioned solve of a netlist with voltage sources needs their "
                                      "elimination (eliminate_sources=False)")
        if reason:
            raise NotImplementedError(f"row-partitioned solve of a netlist with voltage sources: {reason}")
        self.circuit, self.dev, self.table = circuit, dev, table
        self.rank, self.world = int(rank), int(world)
        self.solver = ndist.shared_solver(dev, rank, world)
        m, n, kcl = len(table), table.n, table.kcl
        self.nshare = m * (rank + 1) // world - m * rank // world
        self.stats = {}
        t0 = time.perf_counter()
        self.share = ndist.upload_share(dev, table, _COLUMNS, rank, world)
        self.stats["upload_ms"] = dev.ms_since(t0)
        t0 = time.perf_counter()
        self.bounds = ndist.partition_rows(n, world)
        local, cnt = ndist.exchange_rows(dev, self.share, self.nshare, self.bounds, rank, world,
                                         lambda cols, k, rb, re: dev.select_mna_rows(cols, k, kcl, rb, re))
        csr, rhs = dev.assemble_csr_raw(local, cnt, kcl, n, coo_stride(table))
        self.G, self.A = _rows_of(dev, csr, rhs, self.bounds, rank)
        del csr, local
        self.nnz_full = self._sum_int(self.G.nnz)
        self.stats["full_assemble_ms"] = dev.ms_since(t0)

    def _sum_int(self, v):
        if self.world == 1:
            return int(v)
        import torch
        import torch.distributed as dist
        t = torch.tensor([int(v)], dtype=torch.int64, device=self.dev.dev)
        dist.all_reduce(t)
        return int(t.item())

    def e_table(self):
        """The E rows of every share, in global order, on every rank: (columns, count)."""
        dev = self.dev
        mine, cnt = dev.select_type(self.share, self.nshare, K.T_E)
        cols, total, _ = _allgather(dev, mine, cnt, self.world)
        return cols, total

    def forest(self):
        """(info, forest, E-only columns) of the replicated forest.  The forest's erow, adj_row and
        parent_edge index the E-only table."""
        etab, ne = self.e_table()
        t = self.table
        info, forest = self.dev.source_forest(etab, ne, t.kcl, t.be)
        return info, forest, etab

    def reduced_rows(self, forest, m, stats):
        """The rank's rows of the reduced system over partition_rows(m, world): (LocalRows, rhs).
        stats receives reduced_components (all ranks), reduce_ms and assemble_ms (exchange and build)."""
        dev = self.dev
        t0 = time.perf_counter()
        red, nred = dev.source_reduce(self.share, self.nshare, self.table.kcl, forest)
        stats["reduce_ms"] = dev.ms_since(t0)
        stats["reduced_components"] = self._sum_int(nred)
        if m == 0:
            stats["assemble_ms"] = 0.0
            return None, None
        t0 = time.perf_counter()
        bounds = ndist.partition_rows(m, self.world)
        local, cnt = ndist.exchange_rows(dev, red, nred, bounds, self.rank, self.world, dev.select_local)
        csr, rhs = dev.assemble_csr_raw(local, cnt, m, m, 4)          # stride of R rows (A rows need 2)
        rows, rhs = _rows_of(dev, csr, rhs, bounds, self.rank)
        stats["assemble_ms"] = dev.ms_since(t0)
        return rows, rhs

    def expand(self, info, forest, etab, y):
        """x (n, every rank) from the whole reduced solution y."""
        dev, t = self.dev, self.table
        rb, re = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        x = dev.source_potentials(t.kcl, t.n, forest, y)
        row, rhs, gx = dev.source_tree_rows(t.kcl, t.n, self.nnz_full, rb, re, forest, self.G, self.A, x)
        tree, ntree, _ = _allgather(dev, dict(row=row, rhs=rhs, gx=gx), int(row.numel()), self.world)
        dev.source_currents(t.kcl, etab, forest, info, tree["row"][:ntree], tree["rhs"][:ntree], tree["gx"][:ntree], x)
        return x

    def relres(self, x):
        """||A - G x|| / ||A|| of the full system: the ranks' sums of squares added in rank order."""
        dev = self.dev
        rr, bb = dev.source_residual(self.table.n, self.nnz_full, self.G, self.A, x)
        if self.world > 1:
            import torch
            import torch.distributed as dist
            mine = torch.tensor([rr, bb], dtype=torch.float64, device=dev.dev)
            every = torch.empty(2 * self.world, dtype=torch.float64, device=dev.dev)
            dist.all_gather_into_tensor(every, mine)
            parts = every.cpu().numpy().reshape(self.world, 2)
            rr, bb = 0.0, 0.0
            for k in range(self.world):
                rr, bb = rr + float(parts[k, 0]), bb + float(parts[k, 1])
        return float(np.sqrt(rr / bb) if bb > 0.0 else np.sqrt(rr))

    def solve(self):
        """(x, info): x the whole solution on every rank, info the reduced solve's plus
        info["reduction"] (the single-GPU keys, world and the build's upload_ms / full_assemble_ms)."""
        dev, t = self.dev, self.table
        torch = dev.torch
        stats = dict(world=self.world, **self.stats)
        t0 = time.perf_counter()
        finfo, forest, etab = self.forest()
        stats.update(eliminated=False, sources=finfo["sources"], supernodes=finfo["floating_trees"],
                     grounded_nodes=finfo["grounded_nodes"], forest_ms=dev.ms_since(t0))
        reason = sources.forest_reason(finfo)
        if reason:
            raise NotImplementedError(f"row-partitioned solve of a netlist with voltage sources: {reason}")
        m = finfo["rows"]
        stats.update(eliminated=True, reduced_rows=m, forest_depth=finfo["depth"])
        rows, rhs = self.reduced_rows(forest, m, stats)
        if m > 0:
            t0 = time.perf_counter()
            y_local, info = ndist.amg_then_jacobi(self.solver, rows, rhs, self.circuit.opts)
            stats["solve_ms"] = dev.ms_since(t0)
            y, _, _ = _allgather(dev, dict(y=y_local), int(y_local.numel()), self.world)
            y = y["y"]
            del rows, rhs
        else:                                   # every node is held by a source tree that holds ground
            y = dev.zeros(2, torch.float64)
            info = dict(solver="none", status=0, iterations=0, relres=0.0)
            stats["solve_ms"] = 0.0
        t0 = time.perf_counter()
        x = self.expand(finfo, forest, etab, y)
        stats["expand_ms"] = dev.ms_since(t0)
        t0 = time.perf_counter()
        stats["relres_full"] = self.relres(x)
        stats["relres_ms"] = dev.ms_since(t0)
        return x, dict(info, reduction=stats)
