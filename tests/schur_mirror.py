"""numpy / scipy statement of the Schur-complement solve of nodal_b200/schur.py (csrc/schur.cu).

G = [[L, B], [C, D]] is the sorted MNA matrix (kcl node rows, m branch rows).  split() takes L and
the B lists from the node rows, columns() forms S = D - C Z for Z = L^-1 B, and solve() runs the
refinement x += M^-1 (b - G x) from x = 0 with the block inverse M^-1 (two L solves and one solve
with S).  Every row sum is taken in CSR order with one rounded product and one rounded add per
entry, as csrc/schur_core.cuh does, so the rules can be compared bit for bit.
"""
import numpy as np
import scipy.linalg as sla
import scipy.sparse as sps
import scipy.sparse.csgraph as csgraph
import scipy.sparse.linalg as spla

from nodal_b200 import constants as K


def split(indptr, indices, data, kcl):
    """(L indptr, indices, data), (B ptr, col, val) of the node rows of the sorted CSR."""
    end = int(indptr[kcl])
    rows = np.repeat(np.arange(kcl), np.diff(indptr[: kcl + 1]))
    low = indices[:end] < kcl
    l_ptr = np.zeros(kcl + 1, np.int32)
    b_ptr = np.zeros(kcl + 1, np.int32)
    np.cumsum(np.bincount(rows[low], minlength=kcl), out=l_ptr[1:])
    np.cumsum(np.bincount(rows[~low], minlength=kcl), out=b_ptr[1:])
    return ((l_ptr, indices[:end][low].astype(np.int32), data[:end][low].copy()),
            (b_ptr, (indices[:end][~low] - kcl).astype(np.int32), data[:end][~low].copy()))


def row_dot(ptr, cols, vals, rows, z, limit):
    """For each row of `rows`: the sum over its entries with column < limit of value * z[column],
    entry by entry in CSR order."""
    rows = np.asarray(rows)
    begin, length = ptr[rows].astype(np.int64), (ptr[rows + 1] - ptr[rows]).astype(np.int64)
    acc = np.zeros(len(rows))
    for q in range(int(length.max()) if len(rows) else 0):
        live = np.flatnonzero(length > q)
        p = begin[live] + q
        c = cols[p]
        use = c < limit
        live, p, c = live[use], p[use], c[use]
        acc[live] = acc[live] + vals[p] * z[c]
    return acc


def rhs_batch(Bl, kcl, j0, K_):
    """(K, kcl): the branch columns j0 .. j0 + K - 1 of B."""
    b_ptr, b_col, b_val = Bl
    out = np.zeros((K_, kcl))
    rows = np.repeat(np.arange(kcl), np.diff(b_ptr))
    sel = (b_col >= j0) & (b_col < j0 + K_)
    out[b_col[sel] - j0, rows[sel]] = b_val[sel]
    return out


def columns(indptr, indices, data, kcl, m, j0, Z):
    """S[:, j0 : j0 + K] = D - C Z (m x K)."""
    rows = np.arange(kcl, kcl + m)
    out = np.empty((m, len(Z)))
    for k, z in enumerate(Z):
        d = np.zeros(m)
        for r in range(m):
            p = np.arange(indptr[kcl + r], indptr[kcl + r + 1])
            hit = p[indices[p] == kcl + j0 + k]
            if len(hit):
                d[r] = data[hit[-1]]
        out[:, k] = d - row_dot(indptr, indices, data, rows, z, kcl)
    return out


def branch_rhs(indptr, indices, data, kcl, m, r, t):
    return r[kcl:] - row_dot(indptr, indices, data, np.arange(kcl, kcl + m), t, kcl)


def node_rhs(Bl, kcl, r, xb):
    b_ptr, b_col, b_val = Bl
    return r[:kcl] - row_dot(b_ptr, b_col, b_val, np.arange(kcl), xb, 1 << 62)


def residual(indptr, indices, data, rhs, x):
    n = len(rhs)
    return rhs - row_dot(indptr, indices, data, np.arange(n), x, n)


def r_grounded(table):
    """Every node reaches ground (node kcl) through the R rows alone."""
    kcl = table.kcl
    r = table.type == K.T_R
    a = np.where(table.a[r] < 0, kcl, table.a[r])
    b = np.where(table.b[r] < 0, kcl, table.b[r])
    adj = sps.coo_matrix((np.ones(len(a)), (a, b)), shape=(kcl + 1, kcl + 1))
    _, labels = csgraph.connected_components(adj, directed=False)
    return bool(np.all(labels == labels[kcl]))


def solve(G, rhs, kcl, rtol=1e-10, refine=5, noise=0.0, seed=0):
    """x, info of G x = rhs (G: scipy CSR of the sorted MNA matrix) through the Schur complement.
    noise: relative error put on every L solve (a model of an iterative L solve)."""
    G = sps.csr_matrix(G)
    G.sort_indices()
    indptr, indices, data = G.indptr.astype(np.int64), G.indices.astype(np.int64), G.data
    n = G.shape[0]
    m = n - kcl
    Lc, Bl = split(indptr, indices, data, kcl)
    L = sps.csr_matrix((Lc[2], Lc[1], Lc[0]), shape=(kcl, kcl)).tocsc()
    exact = spla.factorized(L)
    rng = np.random.default_rng(seed)

    def lsolve(b):
        z = exact(b)
        return z * (1 + noise * rng.standard_normal(z.shape)) if noise else z

    S = np.empty((m, m))
    for j0 in range(0, m, 8):
        K_ = min(8, m - j0)
        Z = np.array([lsolve(b) for b in rhs_batch(Bl, kcl, j0, K_)])
        S[:, j0:j0 + K_] = columns(indptr, indices, data, kcl, m, j0, Z)
    lu = sla.lu_factor(S)
    x = np.zeros(n)
    history, reason, step = [], "", 0
    bnorm = np.linalg.norm(rhs)
    while True:
        r = residual(indptr, indices, data, rhs, x)
        relres = np.linalg.norm(r) / bnorm if bnorm > 0 else 0.0
        history.append(relres)
        if relres <= rtol:
            break
        if step == refine:
            reason = "refine"
            break
        if step >= 1 and not relres <= 0.5 * history[-2]:
            reason = "halve"
            break
        t = lsolve(r[:kcl])
        xb = sla.lu_solve(lu, branch_rhs(indptr, indices, data, kcl, m, r, t))
        xn = lsolve(node_rhs(Bl, kcl, r, xb))
        x[:kcl] += xn
        x[kcl:] += xb
        step += 1
    return x, dict(history=history, steps=step, reason=reason, S=S, L=(Lc, Bl))
