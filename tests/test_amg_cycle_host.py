"""CPU checks of the fused V-cycle sweeps (csrc/amg_cycle_core.cuh compiled for the host): on the
hierarchies of the numpy statement (tests/amg_mirror.py), the cycle that forms x0 and the prolongated
iterate at every gathered column equals the cycle that stores them, bit for bit, and both equal the
statement's AMG.cycle to rounding."""
import numpy as np
import pytest
import scipy.sparse as sps

import amg_mirror as mirror
from amg_cycle_host import amg_cycle_host_lib, cycle
from test_amg_host import grid_matrix, random_network


def case(name):
    if name.startswith("grid"):
        return mirror.AMG(grid_matrix(int(name[4:]))[0])
    if name == "random":
        return mirror.AMG(random_network(20000, 60000, 0))
    if name == "jacobi_coarsest":     # more levels, Jacobi on the coarsest level instead of the inverse
        return mirror.AMG(grid_matrix(60)[0], passes=1, direct_max=1, coarse=64)
    # conductances over 8 decades, coarsened down to 64 rows
    return mirror.AMG(random_network(3000, 9000, 7, decades=4.0), coarse=64)


@pytest.mark.parametrize("name", ["grid40", "grid96", "random", "jacobi_coarsest", "random_wide"])
def test_fused_cycle_equals_unfused_bit_for_bit(name):
    M = case(name)
    assert len(M.levels) >= 1
    r = np.random.default_rng(5).standard_normal(M.rows[0])
    z_unfused = cycle(M, r, fused=False)
    z_fused = cycle(M, r, fused=True)
    assert np.array_equal(z_fused.view(np.uint64), z_unfused.view(np.uint64))
    want = M.cycle(r)
    assert np.linalg.norm(z_fused - want) <= 1e-12 * np.linalg.norm(want)


def test_rules_round_once_where_the_kernels_do():
    """x0 = (omega d) b in two roundings, x~ = fma(s, xc, x0), y = fma(omega d, b - acc, x): values
    where a contracted or reassociated form would differ in the last bit."""
    lib = amg_cycle_host_lib()
    ip = np.array([0, 1], dtype=np.int32)
    ix = np.array([0], dtype=np.int32)
    dv = np.array([1.0 + 2.0**-30])
    dinv = np.array([1.0 / 3.0])
    b = np.array([1.0 + 2.0**-27])
    om, sc = 0.8, 1.8
    x = np.empty(1)
    lib.amgc_jacobi0_host(1, dinv.ctypes.data, b.ctypes.data, om, x.ctypes.data)
    assert x[0] == (om * dinv[0]) * b[0]
    xc = np.array([0.1 + 2.0**-40])
    agg = np.zeros(1, dtype=np.int32)
    y = np.empty(1)
    lib.amgc_fused_sweep_host(2, 1, ip.ctypes.data, ix.ctypes.data, dv.ctypes.data, dinv.ctypes.data, b.ctypes.data,
                              om, agg.ctypes.data, xc.ctypes.data, sc, y.ctypes.data)
    from fractions import Fraction as F

    def rnd(q):
        return float(q)

    xa = rnd(F(sc) * F(xc[0]) + F(x[0]))
    acc = rnd(F(dv[0]) * F(xa))
    want = rnd(F(rnd(F(om) * F(dinv[0]))) * F(b[0] - acc) + F(xa))
    assert y[0] == want
