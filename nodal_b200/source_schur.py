"""Sparse solve of netlists with ideal voltage sources and op-amps / dependent sources: the E rows are
eliminated through their forest (sources.py), then the Schur complement of the remaining dependent
branch rows (schur.py) solves the reduced system.

A sheet held at its supply by ideal pads may reach ground only through E rows: the Schur solve of the
full system cannot take it (its L would be singular), and where it can, every pad is a row of S.  The
elimination alone refuses dependent sources.  Here the forest is built on the E rows alone; every node's potential is y[rep_row] + offset
(y = 0 in ground's tree) and the reduced system has the m_n reduced node rows plus one row per
dependent branch (m_d, in branch order).  Its node-node block is the reduced Laplacian of today's
elimination, bit for bit; the other entries come from the rows of the full MNA matrix
(csrc/sources_core.cuh src_dep_row, tests/source_schur_mirror.py).  The unchanged Schur solve of
schur.py runs on it (AMG on L_red, ceil(m_d / 8) batches of L solves instead of one per 8 branch
rows of the full system, dense LU of S, refinement to rtol on the reduced system), and the expansion
recovers the potentials, the dependent currents and the E currents of the full system.

Circuit(netlist, sparse=True, schur=True, eliminate_sources=True) takes this path on a table with E
rows and dependent rows when it qualifies: every R positive, the E rows a forest, no VCVS / VCCS /
CCVS with both output leads in one source tree, every reduced node reaching ground through the
reduced R rows, and 1 <= m_d <= schur_max_branches.  Otherwise, or when the refinement misses rtol,
today's schur=True path runs and Solution.stats["reduction"]["reason"] says why.
"""
from __future__ import annotations

import time

from . import _lib
from . import constants as K
from . import schur
from . import sources

_DEP = (1 << K.T_VCVS) | (1 << K.T_VCCS) | (1 << K.T_CCVS) | (1 << K.T_CCCS)


def applies(circuit):
    """The combined path is asked for: schur=True and eliminate_sources=True on a table with E rows
    and dependent rows."""
    t = circuit.table
    return (circuit.sparse and circuit._dist is None and circuit._schur and circuit._eliminate is True
            and t.has_type(K.T_E) and bool(t.facts()["present"] & _DEP))


def skip_reason(table):
    """What the host can tell before the forest ("" when nothing)."""
    f = table.facts()
    if f["unknown_type"]:
        return "unknown component type"
    if f["r_nonpositive"]:
        return "a resistance is not positive (the reduced L would not be SPD)"
    return ""


def e_forest(dev, dtab, ncomp, kcl):
    """(info, forest, E-only columns) of the forest of the E rows of a mixed table.  With every branch
    owned by one component (nodal_source_dep_map), the E rows' branches renumbered by position are the
    forest's input; the E-only columns keep the table's branch numbers for the expansion."""
    torch = dev.torch
    etab, ne = dev.select_type(dtab, ncomp, K.T_E)
    pos = torch.arange(max(1, ne), dtype=torch.int32, device=dev.dev)
    info, forest = dev.source_forest(dict(etab, branch=pos), ne, kcl, ne)
    return info, forest, etab


def solve(circuit):
    """(x, info) of the full system, or (None, stats) when the path does not apply (stats None) or
    declines (stats["reason"] says why)."""
    if not applies(circuit):
        return None, None
    table, dev, opts = circuit.table, circuit._dev, circuit.options
    kcl, be, ncomp = table.kcl, table.be, len(table)
    max_branches = int(opts.get("schur_max_branches", 8192))
    stats = dict(eliminated=False, applied=False)
    reason = skip_reason(table)
    if reason:
        return None, dict(stats, reason=reason)
    if getattr(circuit, "_G_sorted", None) is not None:     # as in Circuit._device_solve
        circuit.G, circuit._G_sorted = circuit._G_sorted, None
    dtab = circuit._dtab
    ms = sources._ms

    # ---- forest of the E rows alone, the dependent branches numbered in branch order
    t0 = time.perf_counter()
    d_map, md, conflicts = dev.source_dep_map(dtab, ncomp, be)
    stats["dependent_rows"] = md
    if conflicts:
        stats.update(reason="branch rows not owned by exactly one component (duplicate names)", forest_ms=ms(t0, dev))
        return None, stats
    if md > max_branches:
        stats.update(reason=f"{md} dependent branch rows > schur_max_branches ({max_branches})", forest_ms=ms(t0, dev))
        return None, stats
    finfo, forest, etab = e_forest(dev, dtab, ncomp, kcl)
    stats.update(sources=finfo["sources"], supernodes=finfo["floating_trees"], grounded_nodes=finfo["grounded_nodes"])
    reason = sources.forest_reason(finfo)
    if not reason and dev.source_dep_check(dtab, ncomp, kcl, forest):
        reason = "a VCVS / VCCS / CCVS has both output leads in one source tree (its current is undetermined)"
    stats["forest_ms"] = ms(t0, dev)
    if reason:
        stats["reason"] = reason
        return None, stats

    # ---- reduced system
    t0 = time.perf_counter()
    mn = finfo["rows"]
    red, nred = dev.source_reduce(dtab, ncomp, kcl, forest)
    if mn > 0 and not dev.r_grounded(red, nred, mn):
        stats.update(reason="a reduced node does not reach ground through the reduced resistors "
                            "(L would be singular)", reduced_rows=mn, reduce_ms=ms(t0, dev))
        return None, stats
    stats.update(reduced_rows=mn, reduced_components=nred, forest_depth=finfo["depth"], reduce_ms=ms(t0, dev))
    t0 = time.perf_counter()
    Gr, Ar = dev.source_dep_assemble(red, nred, mn, md, kcl, forest, d_map, circuit.G, circuit.A)
    del red
    stats["assemble_ms"] = ms(t0, dev)

    # ---- the Schur solve of schur.py on the reduced system
    rtol = opts.get("rtol", 1e-10)
    sstats = dict(applied=False, branches=md, node_rows=mn)
    if mn == 0:                                 # every node is in ground's tree: the branch rows alone
        t0 = time.perf_counter()
        y, lu = dev.lu_solve(dev.csr_to_dense(Gr), Ar)
        sstats["factor_ms"] = ms(t0, dev)
        if lu["status"] != 0:
            stats["reason"] = f"the dependent rows are singular (zero pivot {lu['info']})"
            return None, dict(stats, schur=sstats)
        sstats.update(applied=True, reason="")
        info = dict(solver="lu", status=0, iterations=0, relres=None)
    else:
        t0 = time.perf_counter()
        L, B = dev.schur_split(Gr, mn)
        sstats["split_ms"] = ms(t0, dev)
        t0 = time.perf_counter()
        try:
            amg = dev.amg(L, **(opts.get("amg") or {}))
        except _lib.NodalLibraryError as err:
            stats["reason"] = f"AMG setup on the reduced L failed: {err}"
            return None, dict(stats, schur=sstats)
        sstats["amg_setup_ms"] = ms(t0, dev)
        try:
            y, info = schur._solve_with(dev, amg, Gr, Ar, B, mn, md, rtol, opts.get("schur_rtol", rtol),
                                        int(opts.get("schur_refine", 5)), opts.get("maxit"), sstats)
        finally:
            amg.close()
        if y is None:
            stats["reason"] = f"Schur solve of the reduced system: {sstats['reason']}"
            return None, dict(stats, schur=sstats)
        info.pop("schur")
    del Gr, Ar

    # ---- expansion on the full system
    t0 = time.perf_counter()
    x, relres = dev.source_expand_dep(etab, kcl, forest, finfo, d_map, mn, y, circuit.G, circuit.A)
    stats.update(eliminated=True, applied=True, reason="", expand_ms=ms(t0, dev), relres_full=relres)
    info.update(solver="source_schur", relres_full=relres, reduction=stats, schur=sstats)
    return x, info
