"""Sparse solve of R / A / E netlists through the elimination of the voltage sources.

Every independent voltage source fixes a potential difference.  When the E rows form a forest (no
loop of sources), every tree of sources becomes one unknown, the remaining system is a weighted
graph Laplacian (SPD) and the AMG-PCG of the R / A path solves it; potentials and source currents
of the full MNA system are recovered exactly (csrc/sources.cu, tests/sources_mirror.py).  Without
it such netlists go to GMRES with a diagonal preconditioner, which stalls on the zero-diagonal
branch rows: above the dense-LU limit that ends in NaNs.

Circuit(netlist, sparse=True, eliminate_sources=...):
    "auto"  (default) eliminate when the table holds only R, A and E rows, every R is positive, the
            E rows form a forest and the system has more rows than dense_fallback_max_rows;
            smaller systems keep the GMRES / dense-LU path
    True    eliminate at any size (ValueError with dependent sources, unless schur=True: then
            source_schur.py eliminates the E rows and solves the rest through the Schur complement);
            a table that does not qualify keeps the existing path, and Solution.stats["reduction"]
            says why
    False   the existing path
"""
from __future__ import annotations

import time

from . import constants as K

_RAE = (1 << K.T_R) | (1 << K.T_A) | (1 << K.T_E)


def skip_reason(table, mode, dense_limit):
    """None: no elimination to consider (no E rows, or switched off); "": eliminate; else why not."""
    if mode is False or not table.has_type(K.T_E):
        return None
    f = table.facts()
    if f["unknown_type"] or f["present"] & ~_RAE:       # "auto", or True with schur=True (source_schur.py)
        return None
    if f["r_nonpositive"]:
        return "a resistance is not positive (the reduced system would not be SPD)"
    if mode == "auto" and table.n <= dense_limit:
        return f"{table.n} rows <= dense_fallback_max_rows ({dense_limit}): the GMRES / dense-LU path is kept"
    return ""


def forest_reason(finfo):
    """Why the forest of csrc/sources.cu cannot eliminate the sources ("" when it can)."""
    if finfo["branch_conflicts"]:
        return "branch rows not owned by exactly one E row (duplicate names)"
    if finfo["loops"]:
        return f"the E rows are not a forest ({finfo['loops']} loop(s); parallel sources or both leads on one node count)"
    return ""


def solve(circuit):
    """(x, info) of the full system through the elimination of a table skip_reason lets through, or
    (None, stats) when the forest declines it (stats["reason"] says why)."""
    table, dev, opts, dtab = circuit.table, circuit._dev, circuit.opts, circuit._dtab
    t0 = time.perf_counter()
    finfo, forest = dev.source_forest(dtab, len(table), table.kcl, table.be)
    stats = dict(eliminated=False, sources=finfo["sources"], supernodes=finfo["floating_trees"],
                 grounded_nodes=finfo["grounded_nodes"], forest_ms=dev.ms_since(t0))
    reason = forest_reason(finfo)
    if reason:
        stats["reason"] = reason
        return None, stats
    t0 = time.perf_counter()
    red, nred = dev.source_reduce(dtab, len(table), table.kcl, forest)
    m = finfo["rows"]
    stats.update(eliminated=True, reduced_rows=m, reduced_components=nred, forest_depth=finfo["depth"],
                 reduce_ms=dev.ms_since(t0))
    torch = dev.torch
    t0 = time.perf_counter()
    if m > 0:
        G, rhs = dev.assemble_csr_raw(red, nred, m, m, 4)          # stride of R rows (A rows need 2)
        stats["assemble_ms"] = dev.ms_since(t0)
        warm = None
        if opts.x0 is not None:
            warm = dev.to_device(opts.x0[forest["roots"][:m].cpu().numpy()])   # roots sit at offset 0
        t0 = time.perf_counter()
        y, info = circuit._spd_solve(G, rhs, opts.spd_solver, opts.spd_rtol, warm)
        stats["solve_ms"] = dev.ms_since(t0)
        del G, rhs
    else:                                       # every node is held by a source tree that holds ground
        y = dev.zeros(2, torch.float64)
        info = dict(solver="none", status=0, iterations=0, relres=0.0)
        stats["assemble_ms"] = stats["solve_ms"] = 0.0
    t0 = time.perf_counter()
    x, relres = dev.source_expand(dtab, table.kcl, forest, finfo, y, circuit.G, circuit.A)
    stats.update(expand_ms=dev.ms_since(t0), relres_full=relres)
    return x, dict(info, reduction=stats)
