"""CPU checks of the Schur-complement solve: the numpy statement (schur_mirror.py) against the oracle,
csrc/schur_core.cuh compiled for the host against the statement bit for bit, the eligibility rules,
the amplifier_grid generator and the CLI flag."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sps

import schur_mirror as mirror
from helpers import block_err, golden, reduce_triples, stamp_on_host, write_csv
from schur_host import schur_host_lib
import nodal_b200 as n
from nodal_b200 import constants as K
from nodal_b200 import generators as gen
from nodal_b200 import schur
from nodal_b200.device import coo_stride
from oracle import mna_oracle as orc

DOC = golden("doc_netlists.json")
# doc / corner netlists with branch rows whose nodes all reach ground through resistors
DOC_SCHUR = ["1.6.1.csv", "opmodel_amplifier.csv", "x_cccs_mixed.csv", "x_ccvs_overwrite.csv",
             "x_vcvs_null_control.csv", "x_vcvs_shared_control.csv"]
# with branch rows, but a node is held by sources alone: the existing path keeps them
DOC_FLOATING = ["buffer.csv", "opmodel_voltage_buffer.csv", "test_1.csv"]


def table_of(rows, tmp_path):
    return n.Netlist(write_csv(rows, tmp_path / "net.csv")).table()


def device_csr(table):
    """The sorted CSR and rhs the device assembles, computed with the host compilation of the stamp."""
    rows, cols, vals = stamp_on_host(table, coo_stride(table))
    indptr, indices, data, rhs = reduce_triples(rows, cols, vals, table.n)
    return indptr, indices, data, rhs


def test_doc_selection(tmp_path):
    """DOC_SCHUR is exactly the doc netlists with branch rows that qualify."""
    picked = []
    for name, d in DOC.items():
        try:
            table = table_of(d["rows"], tmp_path)
        except Exception:          # netlists the reference itself refuses
            continue
        if schur.skip_reason(table, 8192) == "" and mirror.r_grounded(table):
            picked.append(name)
    assert sorted(picked) == sorted(DOC_SCHUR)


@pytest.mark.parametrize("name", DOC_SCHUR)
def test_statement_matches_oracle_doc(name, tmp_path):
    d = DOC[name]
    table = table_of(d["rows"], tmp_path)
    assert table.be > 0 and schur.skip_reason(table, 8192) == "" and mirror.r_grounded(table)
    onet, G, A, _, want = orc.solve_rows(d["rows"], sparse=True, backend="dict")
    x, info = mirror.solve(G.tocsr(), np.asarray(A, float), table.kcl, rtol=1e-10)
    assert not info["reason"], info
    assert block_err(x, want, table.kcl) <= 1e-10


def test_statement_refines_c3(tmp_path):
    """Op-amp gains make S badly conditioned: one application of the block inverse is not enough, a
    few refinement steps are, also when the L solves carry 1e-10 relative noise (the model of the
    AMG solves)."""
    rows = gen.random_opamp_network_rows(M=3968, P=256, S=256, V=64)
    table = table_of(rows, tmp_path)
    assert table.be == 576 and mirror.r_grounded(table)
    onet, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    A = np.asarray(A, float)
    x, info = mirror.solve(G.tocsr(), A, table.kcl, rtol=1e-11, refine=5)
    assert np.linalg.cond(info["S"]) > 1e8
    assert info["history"][1] > 1e-9 and not info["reason"] and info["steps"] == 2, info["history"]
    assert block_err(x, want, table.kcl) <= 1e-9
    x, info = mirror.solve(G.tocsr(), A, table.kcl, rtol=1e-11, refine=5, noise=1e-10)
    assert not info["reason"] and info["steps"] <= 4, info["history"]
    assert block_err(x, want, table.kcl) <= 1e-9
    # without refinement the same netlist is refused, the rule schur.py applies on the device
    _, info = mirror.solve(G.tocsr(), A, table.kcl, rtol=1e-11, refine=1)
    assert info["reason"] == "refine"


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


CORE_CASES = DOC_SCHUR + DOC_FLOATING + ["c3"]


@pytest.mark.parametrize("case", CORE_CASES)
def test_core_matches_statement_bit_for_bit(case, tmp_path):
    rows = gen.random_opamp_network_rows(M=300, P=20, S=20, V=8) if case == "c3" else DOC[case]["rows"]
    table = table_of(rows, tmp_path)
    kcl, m, nn = table.kcl, table.be, table.n
    indptr, indices, data, rhs = device_csr(table)
    indptr, indices = indptr.astype(np.int32), indices.astype(np.int32)
    lib = schur_host_lib()
    # split
    lc, bc = np.zeros(kcl, np.int32), np.zeros(kcl, np.int32)
    lib.schur_counts_host(kcl, _p(indptr), _p(indices), _p(lc), _p(bc))
    (l_ptr, l_idx, l_val), (b_ptr, b_col, b_val) = mirror.split(indptr, indices, data, kcl)
    assert np.array_equal(np.diff(l_ptr), lc) and np.array_equal(np.diff(b_ptr), bc)
    # L is the resistor Laplacian: the CSR of the R rows alone
    rsel = table.type == K.T_R
    rt = n.nodal.ComponentTable(table.type[rsel], table.value[rsel], table.a[rsel], table.b[rsel], kcl=kcl, be=0)
    ri, rx, rd, _ = reduce_triples(*stamp_on_host(rt, 4), kcl)
    assert np.array_equal(ri, l_ptr) and np.array_equal(rx, l_idx) and rd.tobytes() == l_val.tobytes()
    # columns, couplings and residual on random inputs
    rng = np.random.default_rng(7)
    S = np.full((m, m), np.nan)
    want = np.full((m, m), np.nan)
    for j0 in range(0, m, 8):
        K_ = min(8, m - j0)
        Z = np.ascontiguousarray(rng.standard_normal((K_, kcl)))
        lib.schur_columns_host(kcl, m, j0, K_, _p(indptr), _p(indices), _p(data), _p(Z), _p(S))
        want[:, j0:j0 + K_] = mirror.columns(indptr, indices, data, kcl, m, j0, Z)
    assert S.tobytes() == want.tobytes()
    r, t, xb = rng.standard_normal(nn), rng.standard_normal(kcl), rng.standard_normal(m)
    out = np.empty(m)
    lib.schur_branch_rhs_host(kcl, m, _p(indptr), _p(indices), _p(data), _p(r), _p(t), _p(out))
    assert out.tobytes() == mirror.branch_rhs(indptr, indices, data, kcl, m, r, t).tobytes()
    out = np.empty(kcl)
    lib.schur_node_rhs_host(kcl, _p(b_ptr), _p(b_col), _p(b_val), _p(r), _p(xb), _p(out))
    assert out.tobytes() == mirror.node_rhs((b_ptr, b_col, b_val), kcl, r, xb).tobytes()
    x = rng.standard_normal(nn)
    out = np.empty(nn)
    lib.schur_residual_host(nn, _p(indptr), _p(indices), _p(data), _p(rhs), _p(x), _p(out))
    assert out.tobytes() == mirror.residual(indptr, indices, data, rhs, x).tobytes()
    # the statement's split agrees with the full matrix
    G = sps.csr_matrix((data, indices, indptr), shape=(nn, nn)).toarray()
    L = sps.csr_matrix((l_val, l_idx, l_ptr), shape=(kcl, kcl)).toarray()
    B = np.zeros((kcl, m))
    B[np.repeat(np.arange(kcl), np.diff(b_ptr)), b_col] = b_val
    assert np.array_equal(G[:kcl, :kcl], L) and np.array_equal(G[:kcl, kcl:], B)
    assert np.array_equal(mirror.rhs_batch((b_ptr, b_col, b_val), kcl, 0, min(8, m)), B[:, :min(8, m)].T)


def test_eligibility_rules(tmp_path):
    base = DOC["opmodel_amplifier.csv"]["rows"]
    table = table_of(base, tmp_path)
    assert schur.skip_reason(table, 8192) == "" and mirror.r_grounded(table)
    assert "schur_max_branches" in schur.skip_reason(table, table.be - 1)
    neg = table_of(base + [["rn", "R", "-2", "2", "g"]], tmp_path)
    assert "not positive" in schur.skip_reason(neg, 8192)
    assert schur.skip_reason(table_of(orc.grid2d_rows(4), tmp_path), 8192) == "no branch rows"
    # a node held only by a source: passes the host rules, refused by the connectivity check
    floating = table_of(base + [["ex", "E", "1", "x", "g"]], tmp_path)
    assert schur.skip_reason(floating, 8192) == "" and not mirror.r_grounded(floating)
    for bad in ("yes", 1, None):
        with pytest.raises(ValueError):
            schur.check_option({"schur": bad}, True, False)
    with pytest.raises(ValueError):
        schur.check_option({"schur": True, "schur_refine": -1}, True, False)
    assert schur.check_option({}, True, True) is False


def test_option_errors_at_construction(tmp_path):
    """schur=True with the dense path or the row-partitioned one is refused before anything runs."""
    net = n.Netlist(write_csv(DOC["opmodel_amplifier.csv"]["rows"], tmp_path / "amp.csv"))
    with pytest.raises(ValueError):
        n.Circuit(net, sparse=False, schur=True)
    with pytest.raises(NotImplementedError):
        n.Circuit(net, sparse=True, distributed=True, schur=True)


def _csv_rows(net):
    """The csv rows of an amplifier_grid netlist (OPMODEL rows collapsed back from their expansion)."""
    t = net.table()
    nodes = list(net.nodenum) + ["g"]
    name_of = lambda i: "g" if i < 0 else nodes[i]                       # noqa: E731
    keys = net.component_keys
    rows, amps = [], []
    for k in range(len(t)):
        key, typ = keys[k], K.TYPE_NAME[int(t.type[k])]
        if key.startswith("q") and "_" in key:
            if key.endswith("_vcvs"):
                amps.append(key[:-5])
            continue
        row = [key, typ, repr(float(t.value[k])), name_of(t.a[k]), name_of(t.b[k])]
        if typ in ("VCVS", "VCCS", "CCVS", "CCCS"):
            row += [name_of(t.c[k]), name_of(t.d[k])]
        if typ in ("CCVS", "CCCS"):
            row.append(keys[t.drv[k]])
        rows.append(row)
    for q in amps:
        kv = keys.index(q + "_vcvs")
        kf = keys.index(q + "_rf")
        rows.append([q, "OPMODEL", repr(float(t.value[kf])), name_of(t.b[kf]), "g", name_of(t.c[kv]),
                     name_of(t.a[kf])])
    return rows


def test_amplifier_grid_matches_csv(tmp_path):
    net = gen.amplifier_grid(12, 5, seed=3, pitch=4, dependents=2)
    t = net.table()
    rows = _csv_rows(net)
    ref = n.Netlist(write_csv(rows, tmp_path / "amp.csv"))
    rt = ref.table()
    for col in ("type", "value", "a", "b", "c", "d", "drv", "branch"):
        assert getattr(rt, col).tobytes() == getattr(t, col).tobytes(), col
    assert (rt.kcl, rt.be) == (t.kcl, t.be) == (144 + 9 + 3 * 5 + 2 * 2, 9 + 5 + 3 * 2)
    assert dict(ref.nodenum) == {k: net.nodenum[k] for k in net.nodenum}
    assert ref.anomnum == dict(net.anomnum) and ref.ground == net.ground == "g"
    assert ref.table_and_currents()[1] == net.table_and_currents()[1]
    assert list(ref.component_keys) == list(net.component_keys)
    # it qualifies, and the statement solves it
    assert schur.skip_reason(t, 8192) == "" and mirror.r_grounded(t)
    onet, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    x, info = mirror.solve(G.tocsr(), np.asarray(A, float), t.kcl, rtol=1e-10)
    assert not info["reason"] and block_err(x, want, t.kcl) <= 1e-10


def test_cli_flag():
    from nodal_b200.cli import circuit_options, make_parser
    p = make_parser("t", "f")
    assert circuit_options(p.parse_args(["x.csv", "-s"])) == {}
    assert circuit_options(p.parse_args(["x.csv", "-s", "--schur"])) == {"schur": True}
    assert circuit_options(p.parse_args(["x.csv", "--schur"])) == {}
