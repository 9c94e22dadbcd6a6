"""Schur-complement solve of netlists with op-amps and dependent sources (nodal_b200/schur.py,
csrc/schur.cu): the split against the R-only assembly and the statement, the device rules against
their host compilation bit for bit, solves against the oracle / scipy / the dense LU, refinement
failure falling back, and the factor / solve split of the dense LU."""
import ctypes as C
import warnings

import numpy as np
import pytest
import scipy.sparse.linalg as spla

import schur_mirror as mirror
from helpers import block_err, golden, write_csv
from schur_host import schur_host_lib
from test_schur_host import DOC_FLOATING, DOC_SCHUR
import nodal_b200 as n
from nodal_b200 import constants as K
from nodal_b200 import generators as gen
from oracle import mna_oracle as orc

pytestmark = pytest.mark.gpu
DOC = golden("doc_netlists.json")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def host(t):
    return t.cpu().numpy()


def test_split_and_rules_bit_for_bit():
    net = gen.amplifier_grid(48, 12, seed=1, pitch=12, dependents=3)
    circuit = n.Circuit(net, sparse=True, schur=True)
    dev, table, G = circuit._dev, circuit.table, circuit.G
    kcl, m, nn = table.kcl, table.be, table.n
    L, B = dev.schur_split(G, kcl)
    # L is bit-identical to the assembly of the R rows alone
    rt, nr = dev.select_type(circuit._dtab, len(table), K.T_R)
    Lr, _ = dev.assemble_csr_raw(rt, nr, kcl, kcl, 4)
    for a, b in ((L.indptr, Lr.indptr), (L.indices, Lr.indices), (L.data, Lr.data)):
        assert host(a).tobytes() == host(b).tobytes()
    # B lists as the statement splits the host copy of G
    gi, gx, gd = host(G.indptr), host(G.indices), host(G.data)
    (_, _, _), (b_ptr, b_col, b_val) = mirror.split(gi, gx, gd, kcl)
    for a, b in ((B["ptr"], b_ptr), (B["col"], b_col), (B["val"], b_val)):
        assert host(a).tobytes() == np.ascontiguousarray(b).tobytes()
    Bl = (b_ptr, b_col, b_val)
    # the columns of S from the device's own Z, against the host rules fed that Z
    lib = schur_host_lib()
    amg = dev.amg(L)
    try:
        S = dev.empty(m * m, dev.torch.float64).view(m, m)
        want = np.full((m, m), np.nan)
        for j0 in range(0, m, 8):
            K_ = min(8, m - j0)
            rhs = dev.schur_rhs_batch(kcl, j0, K_, B)
            assert host(rhs).tobytes() == mirror.rhs_batch(Bl, kcl, j0, K_).tobytes()
            Z, infos = amg.solve_multi(rhs, rtol=1e-10)
            assert all(i["status"] == 0 for i in infos)
            dev.schur_columns(G, kcl, j0, Z, S)
            lib.schur_columns_host(kcl, m, j0, K_, _p(gi), _p(gx), _p(gd), _p(np.ascontiguousarray(host(Z))), _p(want))
        assert host(S).tobytes() == want.tobytes()
    finally:
        amg.close()
    # the couplings and the residual
    rng = np.random.default_rng(5)
    r, t, xb, x = rng.standard_normal(nn), rng.standard_normal(kcl), rng.standard_normal(m), rng.standard_normal(nn)
    got = host(dev.schur_branch_rhs(G, kcl, dev.to_device(r), dev.to_device(t)))
    assert got.tobytes() == mirror.branch_rhs(gi, gx, gd, kcl, m, r, t).tobytes()
    got = host(dev.schur_node_rhs(kcl, B, dev.to_device(r), dev.to_device(xb)))
    assert got.tobytes() == mirror.node_rhs(Bl, kcl, r, xb).tobytes()
    rd = dev.empty(nn, dev.torch.float64)
    rr, bb = dev.schur_residual(G, circuit.A, dev.to_device(x), rd)
    want = mirror.residual(gi, gx, gd, host(circuit.A), x)
    assert host(rd).tobytes() == want.tobytes()
    assert rr == pytest.approx(float(want @ want), rel=1e-12)
    xd = dev.to_device(x)
    dev.schur_add(xd, dev.to_device(r))
    assert host(xd).tobytes() == (x + r).tobytes()


@pytest.mark.parametrize("name", DOC_SCHUR)
def test_doc_netlists(name, tmp_path):
    d = DOC[name]
    net = n.Netlist(write_csv(d["rows"], tmp_path / name))
    sol = n.Circuit(net, sparse=True, schur=True).solve()
    st = sol.stats["schur"]
    assert st["applied"] and sol.stats["solver"] == "schur" and st["relres_full"] <= 1e-10, st
    assert block_err(sol.result, d["result_sparse"], net.nums["kcl"]) <= 1e-9
    # the default (and schur=False) keep today's path, bit for bit
    a = n.Circuit(n.Netlist(write_csv(d["rows"], tmp_path / "a.csv")), sparse=True).solve()
    b = n.Circuit(n.Netlist(write_csv(d["rows"], tmp_path / "b.csv")), sparse=True, schur=False).solve()
    assert "schur" not in a.stats and a.result.tobytes() == b.result.tobytes()


@pytest.mark.parametrize("name", DOC_FLOATING)
def test_floating_node_keeps_todays_path(name, tmp_path):
    d = DOC[name]
    on = n.Circuit(n.Netlist(write_csv(d["rows"], tmp_path / "a.csv")), sparse=True, schur=True).solve()
    off = n.Circuit(n.Netlist(write_csv(d["rows"], tmp_path / "b.csv")), sparse=True).solve()
    st = on.stats["schur"]
    assert not st["applied"] and "ground through resistors" in st["reason"]
    assert on.result.tobytes() == off.result.tobytes()


def test_c3_16384(tmp_path):
    rows = gen.random_opamp_network_rows()
    net = n.Netlist(write_csv(rows, tmp_path / "c3.csv"))
    assert net.nums["kcl"] + net.nums["be"] == 16384
    circuit = n.Circuit(net, sparse=True, schur=True)
    sol = circuit.solve()
    st = sol.stats["schur"]
    assert st["applied"] and st["relres_full"] <= 1e-10, st
    _, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    kcl = net.nums["kcl"]
    assert block_err(sol.result, want, kcl) <= 1e-9
    dev = circuit._dev
    x, info = dev.lu_solve(dev.csr_to_dense(circuit.G), circuit.A)
    assert info["status"] == 0 and block_err(sol.result, host(x), kcl) <= 1e-9
    # no option: today's path, bit for bit as schur=False
    a = n.Circuit(n.Netlist(write_csv(rows, tmp_path / "a.csv")), sparse=True).solve()
    b = n.Circuit(n.Netlist(write_csv(rows, tmp_path / "b.csv")), sparse=True, schur=False).solve()
    assert a.result.tobytes() == b.result.tobytes()


def test_above_dense_limit_against_spsolve():
    net = gen.amplifier_grid(200, 24, seed=2, pitch=50, dependents=4)
    circuit = n.Circuit(net, sparse=True, schur=True)
    assert circuit.table.n > 32768
    sol = circuit.solve()
    st = sol.stats["schur"]
    assert st["applied"] and st["relres_full"] <= 1e-10, st
    G, A = circuit.G.tocsr(), circuit.A_host
    want = spla.spsolve(G.tocsc(), A)
    assert block_err(sol.result, want, circuit.table.kcl) <= 1e-9


def test_amplifier_grid_2048_bitwise_reruns():
    net = gen.amplifier_grid(2048, 256, seed=0)
    results = []
    for _ in range(2):
        circuit = n.Circuit(net, sparse=True, schur=True)
        sol = circuit.solve()
        st = sol.stats["schur"]
        assert st["applied"] and st["relres_full"] <= 1e-10 and st["branches"] == circuit.table.be, st
        results.append(sol.result)
    G, A = circuit.G.tocsr(), circuit.A_host
    assert np.linalg.norm(A - G @ results[0]) <= 1.05e-10 * np.linalg.norm(A)
    assert results[0].tobytes() == results[1].tobytes()


@pytest.mark.parametrize("refine", [0, 1])
def test_failing_refinement_falls_back(refine, tmp_path):
    rows = DOC["opmodel_amplifier.csv"]["rows"]
    on = n.Circuit(n.Netlist(write_csv(rows, tmp_path / "a.csv")), sparse=True, schur=True, schur_refine=refine,
                   schur_rtol=1e-10, rtol=1e-15).solve()
    off = n.Circuit(n.Netlist(write_csv(rows, tmp_path / "b.csv")), sparse=True, rtol=1e-15).solve()
    st = on.stats["schur"]
    assert not st["applied"] and f"after {refine} refinement" in st["reason"] and st["refine_steps"] == refine
    assert on.stats["solver"] != "schur" and on.result.tobytes() == off.result.tobytes()


@pytest.mark.parametrize("size", [1, 300, 1000])
def test_lu_factor_then_solve_is_lu_solve(device, size):
    rng = np.random.default_rng(size)
    M = rng.standard_normal((size, size)) + size * np.eye(size) * (rng.random(size) < 0.5)
    b = rng.standard_normal(size)
    x1, info = device.lu_solve(device.to_device(M), device.to_device(b))
    assert info["status"] == 0
    LU = device.to_device(M)
    ipiv, finfo = device.lu_factor(LU)
    assert finfo["status"] == 0
    x2 = device.lu_solve_factored(LU, ipiv, device.to_device(b))
    assert host(x1).tobytes() == host(x2).tobytes()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert np.allclose(M @ host(x2), b, rtol=0, atol=1e-8 * np.abs(b).max() * max(1.0, np.linalg.cond(M)))
