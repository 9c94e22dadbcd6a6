"""The compact SELL entry encoding (16-bit column offsets, 1-byte indices into a table of distinct
values) computes bit for bit what the wide one (int32 columns, double values; NODAL_SELL_WIDE=1)
computes: the SpMV, one AMG V-cycle, the Jacobi-PCG and the one-rank row-partitioned AMG-PCG, on a grid
and a power-grid Laplacian (compact) and a network of random conductances (wide either way)."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.sparse as sps

from nodal_b200 import _lib
from nodal_b200 import dist as ndist
from nodal_b200.device import DeviceCSR

pytestmark = pytest.mark.gpu


def grid_laplacian(m, g):
    """m x m grid, conductance g[e] on edge e (horizontal edges first), node 0 grounded by 1 S."""
    idx = np.arange(m * m).reshape(m, m)
    a = np.concatenate([idx[:, :-1].ravel(), idx[:-1, :].ravel()])
    b = np.concatenate([idx[:, 1:].ravel(), idx[1:, :].ravel()])
    g = np.broadcast_to(np.asarray(g, dtype=np.float64), a.shape)
    n = m * m
    L = sps.coo_matrix((np.concatenate([-g, -g]), (np.concatenate([a, b]), np.concatenate([b, a]))), shape=(n, n))
    d = np.bincount(a, g, n) + np.bincount(b, g, n)
    d[0] += 1.0
    return sps.csr_matrix(L + sps.diags(d))


def power_grid_laplacian(m, pitch, r):
    """The reduced Laplacian of a supply-pad grid: one resistance r everywhere, the pad nodes (every
    `pitch` nodes in both directions) eliminated; their neighbours keep the conductance to them on the
    diagonal."""
    L = grid_laplacian(m, 1.0 / r).tolil()
    L[0, 0] -= 1.0
    L = L.tocsr()
    pads = np.zeros((m, m), dtype=bool)
    pads[::pitch, ::pitch] = True
    keep = np.flatnonzero(~pads.ravel())
    return sps.csr_matrix(L[keep][:, keep])


CASES = {
    "grid": (lambda: grid_laplacian(96, 1.0), True),
    "power_grid": (lambda: power_grid_laplacian(80, 7, 0.05), True),
    "random": (lambda: grid_laplacian(72, np.random.default_rng(3).uniform(0.5, 2.0, 2 * 72 * 71)), False),
}


def to_device(device, M):
    M = sps.csr_matrix(M)
    M.sort_indices()
    return DeviceCSR(M.shape[0], device.to_device(M.indptr.astype(np.int32)),
                     device.to_device(M.indices.astype(np.int32)), device.to_device(M.data))


def encodings(fn):
    """fn() with the library's choice, then with NODAL_SELL_WIDE=1."""
    os.environ.pop("NODAL_SELL_WIDE", None)
    picked = fn()
    os.environ["NODAL_SELL_WIDE"] = "1"
    try:
        wide = fn()
    finally:
        os.environ.pop("NODAL_SELL_WIDE", None)
    return picked, wide


def sell_spmv(device, csr, x):
    h = C.c_void_p()
    p = device.ptr
    _lib.check(device.lib.nodal_sell_create(device.ctx, csr.n, csr.nnz, p(csr.indptr), p(csr.indices),
                                            p(csr.data), C.byref(h), device.stream()), "sell_create")
    try:
        y = device.empty(csr.n, device.torch.float64)
        _lib.check(device.lib.nodal_sell_spmv(device.ctx, h, p(x), p(y), device.stream()), "sell_spmv")
        return y.cpu().numpy(), int(device.lib.nodal_sell_compact(h)), int(device.lib.nodal_sell_padded_nnz(h))
    finally:
        device.lib.nodal_sell_destroy(h)


@pytest.mark.parametrize("name", sorted(CASES))
def test_sell_spmv_bits(device, name):
    make, compact = CASES[name]
    M = make()
    csr = to_device(device, M)
    x = np.random.default_rng(1).standard_normal(M.shape[0])
    x[::17] = -0.0
    xd = device.to_device(x)
    (y, enc, padded), (yw, encw, paddedw) = encodings(lambda: sell_spmv(device, csr, xd))
    assert enc == int(compact) and encw == 0
    assert padded == paddedw
    assert np.array_equal(y.view(np.uint64), yw.view(np.uint64))
    assert np.max(np.abs(y - M @ x)) <= 1e-12 * np.max(np.abs(M) @ np.abs(x))


@pytest.mark.parametrize("name", sorted(CASES))
def test_amg_apply_bits(device, name):
    M = CASES[name][0]()
    csr = to_device(device, M)
    r = device.to_device(np.random.default_rng(2).standard_normal(M.shape[0]))

    def apply():
        h = device.amg(csr, coarse=64)
        try:
            return h.apply(r).cpu().numpy()
        finally:
            h.close()

    z, zw = encodings(apply)
    assert np.array_equal(z.view(np.uint64), zw.view(np.uint64))


@pytest.mark.parametrize("name", sorted(CASES))
def test_jacobi_pcg_bits(device, name):
    M = CASES[name][0]()
    csr = to_device(device, M)
    b = device.to_device(np.random.default_rng(4).standard_normal(M.shape[0]))
    (x, info), (xw, infow) = encodings(lambda: device.pcg(csr, b, rtol=1e-10))
    assert info["iterations"] == infow["iterations"]
    assert np.array_equal(x.cpu().numpy().view(np.uint64), xw.cpu().numpy().view(np.uint64))


@pytest.mark.parametrize("name", sorted(CASES))
def test_dist_single_rank_amg_pcg_bits(device, name):
    M = CASES[name][0]()
    csr = to_device(device, M)
    n = M.shape[0]
    rhs = device.to_device(np.random.default_rng(5).standard_normal(n))
    bounds = np.array([0, n], dtype=np.int32)
    solver = ndist.single_solver(device)

    def solve():
        x, info = solver.solve_amg(n, bounds, csr.indptr, csr.indices, csr.data, rhs, rtol=1e-10, gather_below=300)
        return x.cpu().numpy(), info

    (x, info), (xw, infow) = encodings(solve)
    assert info["status"] == 0 and info["distributed_levels"] >= 1
    assert info["iterations"] == infow["iterations"]
    assert np.array_equal(x.view(np.uint64), xw.view(np.uint64))


# 255 nonzero values + the +0.0 of the padding fill the 256-entry table, one more goes wide.  "block": all
# rows in one thread block's slices, so its own hash set overflows; "merged": 64 rows per value, so every
# block sees a handful of values and only the merged global set holds them all.
@pytest.mark.parametrize("layout", ["block", "merged"])
@pytest.mark.parametrize("distinct,compact", [(255, True), (256, False)])
def test_table_boundary(device, layout, distinct, compact):
    per = 1 if layout == "block" else 64
    n = distinct * per
    vals = 1.0 + np.arange(n) // per + 0.5 ** 20 * (np.arange(n) // per)
    M = sps.diags(vals).tocsr()
    csr = to_device(device, M)
    x = np.random.default_rng(6).standard_normal(n)
    xd = device.to_device(x)
    (y, enc, _), (yw, encw, _) = encodings(lambda: sell_spmv(device, csr, xd))
    assert enc == int(compact) and encw == 0
    assert np.array_equal(y.view(np.uint64), yw.view(np.uint64))
    assert np.array_equal(y, vals * x)
