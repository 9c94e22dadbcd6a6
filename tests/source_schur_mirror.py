"""numpy statement of the solve of nodal_b200/source_schur.py: the E rows eliminated through their
forest, the dependent branch rows kept (csrc/sources_core.cuh src_dep_row, csrc/sources.cu).

The forest is built on the E rows alone (sources_mirror.forest on the E-only table, its branches
renumbered by position).  The reduced system has the m_n reduced node rows and one row per
dependent branch (m_d, branch order).  Its triples are, in this emission order: the stamp of the
reduced R / A table (component order), then the mapped entries of the full sorted MNA matrix, row by
row in CSR order (node rows outside ground's tree: their dependent branch columns; dependent branch
rows: node columns to rep_row unless in ground's tree, dependent branch columns renumbered, and one
right-hand-side entry A - sum G o over the node columns).  helpers.reduce_triples sums them as the
device's CSR build does, so the result can be compared bit for bit.
"""
from types import SimpleNamespace

import numpy as np
import scipy.sparse as sps
import scipy.sparse.csgraph as csgraph

import sources_mirror as sm
from helpers import reduce_triples

T_R, T_A, T_E = 0, 1, 2
DEP = (3, 4, 5, 6)          # VCVS, VCCS, CCVS, CCCS
COLLAPSE = (3, 4, 5)        # the ones whose branch row carries the incidence of their output leads


def dep_map(table):
    """(d_map over the branches, dependent branch ids in branch order, conflicts)."""
    be = table.be
    own = table.branch >= 0
    used = np.bincount(table.branch[own], minlength=be)[:be]
    dep = np.zeros(be, bool)
    dep[table.branch[own & np.isin(table.type, DEP)]] = True
    d_map = np.where(dep, np.cumsum(dep) - dep, -1).astype(np.int32)
    return d_map, np.flatnonzero(dep), int(np.count_nonzero(used != 1))


def e_table(table, renumber):
    """The E-only table (renumber: its branches by position, as the forest takes them)."""
    e = np.flatnonzero(table.type == T_E)
    return SimpleNamespace(type=table.type[e], value=table.value[e], a=table.a[e], b=table.b[e],
                           branch=np.arange(len(e), dtype=np.int32) if renumber else table.branch[e],
                           kcl=table.kcl, be=len(e) if renumber else table.be, n=table.n)


def forest(table):
    return sm.forest(e_table(table, True))


def collapsed(table, f):
    """VCVS / VCCS / CCVS rows whose output leads share rep_row."""
    kcl = table.kcl
    node = lambda lead: np.where(lead < 0, kcl, lead)            # noqa: E731
    sel = np.isin(table.type, COLLAPSE)
    rep = f["rep_row"]
    return int(np.count_nonzero(rep[node(table.a[sel])] == rep[node(table.b[sel])]))


def r_grounded(typ, a, b, m):
    """Every one of m rows reaches ground (-1) through the R rows of the table (typ, a, b)."""
    r = typ == T_R
    aa, bb = np.where(a[r] < 0, m, a[r]), np.where(b[r] < 0, m, b[r])
    adj = sps.coo_matrix((np.ones(len(aa)), (aa, bb)), shape=(m + 1, m + 1))
    _, labels = csgraph.connected_components(adj, directed=False)
    return bool(np.all(labels == labels[m]))


def reason(table, max_branches=8192):
    """The refusal of source_schur.solve, in its order ("" when the table qualifies)."""
    if np.any(table.value[table.type == T_R] <= 0):
        return "not positive"
    d_map, deps, conflicts = dep_map(table)
    if conflicts:
        return "duplicate names"
    if len(deps) > max_branches:
        return "schur_max_branches"
    f = forest(table)
    if not f["ok"]:
        return "forest"
    if collapsed(table, f):
        return "one source tree"
    typ, val, a, b = sm.reduce_table(table, f)
    if f["rows"] > 0 and not r_grounded(typ, a, b, f["rows"]):
        return "does not reach ground"
    return ""


def stamp_ra(typ, val, a, b, n):
    """Triples of an R / A table's stamp in emission order (col == n: the rhs)."""
    rows, cols, vals = [], [], []
    for t, v, p, q in zip(typ, val, a, b):
        if t == T_R:
            g = 1.0 / v
            out = ([(p, p, g)] if p >= 0 else []) + ([(q, q, g)] if q >= 0 else [])
            if p >= 0 and q >= 0:
                out += [(p, q, -g), (q, p, -g)]
        else:
            out = ([(p, n, v)] if p >= 0 else []) + ([(q, n, -v)] if q >= 0 else [])
        for r, c, x in out:
            rows.append(r), cols.append(c), vals.append(x)
    return np.array(rows, np.int64), np.array(cols, np.int64), np.array(vals, np.float64)


def dep_triples(indptr, indices, data, rhs, kcl, f, d_map, mn, nr):
    """The mapped entries of the full sorted CSR, rows in order, entries in CSR order."""
    rep, off = f["rep_row"], f["offset"]
    rows, cols, vals = [], [], []
    for i in range(len(indptr) - 1):
        p0, p1 = int(indptr[i]), int(indptr[i + 1])
        if i < kcl:
            if rep[i] < 0:
                continue
            for p in range(p0, p1):
                c = int(indices[p])
                if c >= kcl and d_map[c - kcl] >= 0:
                    rows.append(rep[i]), cols.append(mn + d_map[c - kcl]), vals.append(data[p])
            continue
        d = d_map[i - kcl]
        if d < 0:
            continue
        acc = 0.0
        for p in range(p0, p1):
            c = int(indices[p])
            if c < kcl:
                acc = acc + data[p] * off[c]
                if rep[c] >= 0:
                    rows.append(mn + d), cols.append(rep[c]), vals.append(data[p])
            elif d_map[c - kcl] >= 0:
                rows.append(mn + d), cols.append(mn + d_map[c - kcl]), vals.append(data[p])
        rows.append(mn + d), cols.append(nr), vals.append(rhs[i] - acc)
    return np.array(rows, np.int64), np.array(cols, np.int64), np.array(vals, np.float64)


def reduced_system(table, G, A):
    """(f, d_map, deps, mn, md, triples, (indptr, indices, data, rhs)) of the reduced system;
    G the full MNA matrix (scipy), A its rhs."""
    G = sps.csr_matrix(G)
    G.sort_indices()
    f = forest(table)
    assert f["ok"], f["reason"]
    d_map, deps, _ = dep_map(table)
    mn, md = f["rows"], len(deps)
    nr = mn + md
    red = sm.reduce_table(table, f)
    t1 = stamp_ra(*red, nr)
    t2 = dep_triples(G.indptr, G.indices, G.data, np.asarray(A, float), table.kcl, f, d_map, mn, nr)
    triples = tuple(np.r_[x, y] for x, y in zip(t1, t2))
    return f, d_map, deps, mn, md, triples, reduce_triples(*triples, nr), t2


def expand(table, f, deps, mn, xr, G, A):
    """x of the full system: potentials from xr[:mn], the dependent currents xr[mn:], the E currents
    from the subtree sums of rho = A - G [e; x_dep; 0]."""
    kcl = table.kcl
    x = np.zeros(table.n)
    x[:kcl] = sm.potentials(f, xr[:mn], kcl)
    x[kcl + deps] = xr[mn:]
    rho = (np.asarray(A, float) - sps.csr_matrix(G) @ x)[:kcl]
    out = sm.expand(e_table(table, False), f, xr[:mn], rho)
    out[kcl + deps] = xr[mn:]
    return out


def solve(table, G, A):
    """The whole statement: reduced system, dense solve, expansion.  Returns (x, parts)."""
    f, d_map, deps, mn, md, triples, csr, _ = reduced_system(table, G, A)
    indptr, indices, data, rhs = csr
    nr = mn + md
    Gr = sps.csr_matrix((data, indices, indptr), shape=(nr, nr)).toarray()
    xr = np.linalg.solve(Gr, rhs) if nr else np.zeros(0)
    return expand(table, f, deps, mn, xr, G, A), dict(f=f, mn=mn, md=md, Gr=Gr, rhs=rhs, xr=xr)
