"""numpy statement of the voltage-source elimination (csrc/sources.cu, csrc/sources_core.cuh).

Every E row fixes e_a - e_b = V.  When the E rows of an R / A / E table form a forest over the
nodes (ground is node kcl), each tree gets one unknown: its root is ground when the tree holds it
(every potential in it is then known), else its smallest node.  Every node's potential is
y[rep_row] + offset.  The reduced system Z^T G_kk Z y = Z^T (A_k - G_kk v0) is the stamp of an
R / A table over the roots, and the source currents come back from KCL summed over the subtree
each source cuts off.  Orders (reduced rows, reduced table, children of a node) are the device's,
so its outputs can be compared bit for bit.
"""
import numpy as np
import scipy.sparse as sps
import scipy.sparse.csgraph as csgraph

T_R, T_A, T_E = 0, 1, 2
GROUND = -1


def forest(table):
    """dict(ok, reason, sources, loops, branch_conflicts, trees, floating_trees, grounded_nodes, rows,
    depth) and, when ok: rep_row, offset, parent_edge, depth_of, roots, erow (per-node arrays of kcl + 1)."""
    kcl, be = table.kcl, table.be
    node = lambda lead: np.where(lead < 0, kcl, lead)            # noqa: E731
    erow = np.flatnonzero(table.type == T_E)
    ea, eb = node(table.a[erow]), node(table.b[erow])
    out = dict(sources=len(erow), loops=0, branch_conflicts=0, trees=0, floating_trees=0, grounded_nodes=0,
               rows=0, depth=0, ok=False, reason=None)
    if len(erow) != be:
        out["branch_conflicts"] = abs(len(erow) - be)
    else:
        used = np.bincount(table.branch[erow], minlength=be)
        out["branch_conflicts"] = int(np.count_nonzero(used != 1))
    if out["branch_conflicts"]:
        out["reason"] = "branch rows not owned by exactly one E row"
        return out
    nodes = kcl + 1
    g = sps.coo_matrix((np.ones(len(erow)), (ea, eb)), shape=(nodes, nodes))
    _, lab = csgraph.connected_components(g, directed=False)
    # label = smallest node of the component, as the device's union-find leaves it
    first = np.full(lab.max() + 1, nodes, np.int64)
    np.minimum.at(first, lab, np.arange(nodes))
    labels = first[lab]
    deg = np.bincount(np.r_[ea, eb], minlength=nodes)
    touched = deg > 0
    head = touched & (labels == np.arange(nodes))
    out["trees"] = int(head.sum())
    out["loops"] = int(len(erow) - (touched.sum() - out["trees"]))
    out["grounded_nodes"] = int(np.count_nonzero(touched[:kcl] & (labels[:kcl] == labels[kcl])))
    out["floating_trees"] = int(np.count_nonzero(head & (labels != labels[kcl])))
    if out["loops"]:
        out["reason"] = "the E rows form a loop (or an E row has both leads on one node)"
        return out
    root = np.where(labels == labels[kcl], kcl, labels)
    free = (np.arange(nodes) < kcl) & (root == np.arange(nodes))
    red = np.cumsum(free) - free
    rep_row = np.where(root == kcl, GROUND, red[root]).astype(np.int32)
    roots = np.flatnonzero(free).astype(np.int32)
    offset = np.zeros(nodes)
    parent_edge = np.full(nodes, -1, np.int32)
    depth = np.where(root == np.arange(nodes), 0, -1).astype(np.int32)
    # adjacency ordered by (node, other node), as the device sorts it
    hu, hw, hr = np.r_[ea, eb], np.r_[eb, ea], np.r_[erow, erow]
    order = np.lexsort((hw, hu))
    hu, hw, hr = hu[order], hw[order], hr[order]
    level = 0
    while len(erow):
        claim = (depth[hu] == level) & (depth[hw] < 0)
        if not claim.any():
            break
        w, r, u = hw[claim], hr[claim], hu[claim]
        depth[w] = level + 1
        parent_edge[w] = r
        anode = node(table.a[r]) == w
        v = table.value[r]
        offset[w] = np.where(anode, offset[u] + v, offset[u] - v)
        level += 1
    out.update(ok=True, rows=len(roots), depth=level, rep_row=rep_row, offset=offset, parent_edge=parent_edge,
               depth_of=depth, roots=roots, erow=erow.astype(np.int32), adj_node=hu, adj_other=hw)
    return out


def reduce_table(table, f):
    """(type, value, a, b) of the reduced R / A table, component order, up to two rows per component."""
    kcl = table.kcl
    na = np.where(table.a < 0, kcl, table.a)
    nb = np.where(table.b < 0, kcl, table.b)
    ra, rb = f["rep_row"][na], f["rep_row"][nb]
    oa, ob = f["offset"][na], f["offset"][nb]
    t = table.type
    live = ((t == T_R) | (t == T_A)) & (ra != rb)
    extra = live & (t == T_R) & (oa != ob)
    idx = np.r_[np.flatnonzero(live), np.flatnonzero(extra)]
    slot = np.r_[np.zeros(live.sum(), np.int64), np.ones(extra.sum(), np.int64)]
    order = np.argsort(idx * 2 + slot, kind="stable")
    idx, slot = idx[order], slot[order]
    typ = np.where(slot == 1, T_A, t[idx]).astype(np.uint8)
    with np.errstate(divide="ignore", invalid="ignore"):
        val = np.where(slot == 1, -(oa[idx] - ob[idx]) / table.value[idx], table.value[idx])
    return typ, val, ra[idx].astype(np.int32), rb[idx].astype(np.int32)


def potentials(f, y, kcl):
    rep = f["rep_row"][:kcl]
    return np.where(rep < 0, 0.0, y[np.maximum(rep, 0)] if len(y) else 0.0) + f["offset"][:kcl]


def expand(table, f, y, rho):
    """x = [e; i]: potentials from y, source currents from the KCL residual rho (kcl entries) summed
    over every source's subtree, deepest level first, children in node order."""
    kcl, n = table.kcl, table.n
    x = np.zeros(n)
    x[:kcl] = potentials(f, y, kcl)
    acc = np.r_[np.asarray(rho, float), 0.0]
    depth, pe = f["depth_of"], f["parent_edge"]
    node = lambda lead: kcl if lead < 0 else int(lead)            # noqa: E731
    for d in range(f["depth"], 0, -1):
        for w in np.flatnonzero(depth == d):                       # ascending: each parent adds children in order
            r = int(pe[w])
            a, b = node(table.a[r]), node(table.b[r])
            x[kcl + table.branch[r]] = -acc[w] if a == w else acc[w]
            parent = b if a == w else a
            acc[parent] = acc[parent] + acc[w]
    return x


def laplacian(typ, val, a, b, m):
    """Stamp of an R / A table with m rows (scipy; the order of the sums does not matter here)."""
    R = typ == T_R
    g = 1.0 / val[R]
    ra, rb = a[R], b[R]
    i = np.r_[ra, rb, ra, rb]
    j = np.r_[ra, rb, rb, ra]
    v = np.r_[g, g, -g, -g]
    keep = (i >= 0) & (j >= 0)
    G = sps.csr_matrix((v[keep], (i[keep], j[keep])), shape=(m, m))
    rhs = np.zeros(m)
    A = typ == T_A
    np.add.at(rhs, a[A][a[A] >= 0], val[A][a[A] >= 0])
    np.add.at(rhs, b[A][b[A] >= 0], -val[A][b[A] >= 0])
    return G, rhs


def solve(table, G, A):
    """The whole statement on the host: forest, reduced table, spsolve of the reduced Laplacian,
    expansion with rho = A_k - G_k [e; 0] of the full MNA matrix G."""
    import scipy.sparse.linalg as spla
    f = forest(table)
    assert f["ok"], f["reason"]
    m = f["rows"]
    Gr, br = laplacian(*reduce_table(table, f), m)
    y = spla.spsolve(Gr.tocsc(), br) if m else np.zeros(0)
    y = np.atleast_1d(y)
    kcl = table.kcl
    e = np.r_[potentials(f, y, kcl), np.zeros(table.n - kcl)]
    rho = (np.asarray(A) - G @ e)[:kcl]
    return expand(table, f, y, rho), f
