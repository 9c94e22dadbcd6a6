"""CPU checks of the solve with E rows and dependent branch rows (nodal_b200/source_schur.py): the
numpy statement (source_schur_mirror.py) against the oracle, the dependent-row rules of
csrc/sources_core.cuh compiled for the host against the statement bit for bit, the eligibility rules,
the options, amplifier_grid(ideal_pads=True) against its csv and the CLI mapping."""
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg  # noqa: F401  (sps.linalg)

import source_schur_host as host
import source_schur_mirror as mirror
import sources_mirror as sm
from helpers import block_err, golden, reduce_triples, stamp_on_host, write_csv
from test_schur_host import _csv_rows
import nodal_b200 as n
from nodal_b200 import constants as K
from nodal_b200 import generators as gen
from nodal_b200 import schur, source_schur, sources
from oracle import mna_oracle as orc

DOC = golden("doc_netlists.json")
# doc netlists with E rows and dependent rows that qualify (two of them were turned away by the Schur
# solve of the full system because a node is held by a source alone)
DOC_SOURCE_SCHUR = ["1.6.1.csv", "buffer.csv", "opmodel_amplifier.csv", "opmodel_voltage_buffer.csv",
                    "x_cccs_mixed.csv", "x_ccvs_overwrite.csv", "x_vcvs_shared_control.csv"]
# 1e-12 A currents next to 10 V potentials (cond ~1e6): the oracle itself is 5e-6 off in those
# currents, so they are compared whole-vector normwise, as tests/test_oracle.py does
WHOLE_VECTOR = ("buffer.csv", "opmodel_voltage_buffer.csv")

# e1's output lead 2 and control lead 1 lie in one source tree ("ve" ties nodes 1 and 2): in its
# reduced branch row they add up; f1 / h1 are controlled through r2, which leaves that tree
HAND_TREE = [["ve", "E", "0.5", "1", "2"], ["r1", "R", "2", "1", "g"], ["r2", "R", "3", "2", "3"],
             ["r3", "R", "5", "3", "g"], ["r4", "R", "7", "3", "4"], ["r5", "R", "11", "4", "g"],
             ["e1", "VCVS", "2", "2", "4", "1", "3"], ["f1", "CCCS", "0.25", "3", "g", "2", "3", "r2"],
             ["h1", "CCVS", "1.5", "5", "g", "2", "3", "r2"], ["r6", "R", "13", "5", "1"]]
# every node in ground's tree (m_n = 0): the dependent rows alone (only a CCCS can qualify there, the
# output leads of any other dependent source would lie in one tree)
HAND_GROUND = [["va", "E", "1", "1", "g"], ["vb", "E", "2", "2", "1"], ["r1", "R", "4", "1", "2"],
               ["vc", "E", "3", "3", "g"], ["f1", "CCCS", "0.5", "2", "g", "1", "2", "r1"],
               ["r2", "R", "5", "2", "3"], ["f2", "CCCS", "2", "3", "1", "2", "3", "r2"]]


def table_of(rows, tmp_path):
    return n.Netlist(write_csv(rows, tmp_path / "net.csv")).table()


def doc_err(name, x, want, kcl):
    if name in WHOLE_VECTOR:
        want = np.asarray(want, float)
        return np.max(np.abs(np.asarray(x) - want)) / np.max(np.abs(want))
    return block_err(x, want, kcl)


def test_doc_selection(tmp_path):
    """DOC_SOURCE_SCHUR is exactly the doc netlists with E rows and dependent rows that qualify."""
    picked = []
    for name, d in DOC.items():
        try:
            table = table_of(d["rows"], tmp_path)
        except Exception:          # netlists the reference itself refuses
            continue
        f = table.facts()
        if table.has_type(K.T_E) and f["present"] & source_schur._DEP and mirror.reason(table) == "":
            picked.append(name)
    assert sorted(picked) == sorted(DOC_SOURCE_SCHUR)


@pytest.mark.parametrize("name", DOC_SOURCE_SCHUR)
def test_statement_matches_oracle_doc(name, tmp_path):
    d = DOC[name]
    table = table_of(d["rows"], tmp_path)
    _, G, A, _, want = orc.solve_rows(d["rows"], sparse=True, backend="dict")
    x, parts = mirror.solve(table, G.tocsr(), np.asarray(A, float))
    assert parts["md"] >= 1
    assert doc_err(name, x, want, table.kcl) <= 1e-9


@pytest.mark.parametrize("rows,mn,md", [(HAND_TREE, 4, 3), (HAND_GROUND, 0, 2)])
def test_statement_hand_made(rows, mn, md, tmp_path):
    table = table_of(rows, tmp_path)
    assert mirror.reason(table) == ""
    _, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    x, parts = mirror.solve(table, G.tocsr(), np.asarray(A, float))
    assert parts["mn"] == mn and parts["md"] == md
    assert block_err(x, want, table.kcl) <= 1e-12


def test_output_and_control_in_one_tree_sum(tmp_path):
    """e1's output lead 2 (+1) and control lead 1 (-2) map to one reduced column: their entries add
    (-1), where re-stamping the mapped leads would have let the reference's '=' keep one of them."""
    table = table_of(HAND_TREE, tmp_path)
    _, G, A, _, _ = orc.solve_rows(HAND_TREE, sparse=True, backend="dict")
    f, d_map, deps, mn, md, _, (ip, ix, dx, _), t2 = mirror.reduced_system(table, G.tocsr(), np.asarray(A, float))
    Gr = sps.csr_matrix((dx, ix, ip), shape=(mn + md, mn + md)).toarray()
    k = list(n.Netlist(write_csv(HAND_TREE, tmp_path / "net.csv")).component_keys).index("e1")
    row = mn + d_map[table.branch[k]]
    tree = f["rep_row"][table.a[k]]
    assert tree == f["rep_row"][table.c[k]] >= 0
    rows, cols, vals = t2
    hit = (rows == row) & (cols == tree)
    assert sorted(vals[hit].tolist()) == [-2.0, 1.0] and Gr[row, tree] == -1.0


def full_csr(table):
    """The sorted CSR and rhs the device assembles (host compilation of the stamp) as scipy / numpy."""
    from nodal_b200.device import coo_stride
    ip, ix, dx, rhs = reduce_triples(*stamp_on_host(table, coo_stride(table)), table.n)
    return sps.csr_matrix((dx, ix, ip), shape=(table.n, table.n)), rhs


def case_table(case, tmp_path):
    if case == "amp_ideal":
        return gen.amplifier_grid(10, 3, seed=1, pitch=3, dependents=2, ideal_pads=True).table()
    rows = {"hand_tree": HAND_TREE, "hand_ground": HAND_GROUND}.get(case) or DOC[case]["rows"]
    return table_of(rows, tmp_path)


CORE_CASES = DOC_SOURCE_SCHUR + ["hand_tree", "hand_ground", "amp_ideal"]


@pytest.mark.parametrize("case", CORE_CASES)
def test_core_matches_statement_bit_for_bit(case, tmp_path):
    table = case_table(case, tmp_path)
    G, A = full_csr(table)
    f, d_map, deps, mn, md, triples, csr, t2 = mirror.reduced_system(table, G, A)
    nr = mn + md
    got = host.dep_triples(G.indptr, G.indices, G.data, A, table.kcl, f, d_map, mn, nr)
    for a, b in zip(got, t2):
        assert a.tobytes() == b.tobytes()
    # the reduced table's stamp as the device emits it, then the dependent triples: the same CSR
    typ, val, a, b = sm.reduce_table(table, f)
    r1, c1, v1 = stamp_on_host(n.nodal.ComponentTable(typ, val, a, b, kcl=mn, be=md), 4)
    ip, ix, dx, rhs = reduce_triples(np.r_[r1, got[0]], np.r_[c1, got[1]], np.r_[v1, got[2]], nr)
    for x, y in zip((ip, ix, dx, rhs), csr):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes()
    # the node-node block and node rhs are the reduced Laplacian of the elimination, bit for bit
    li, lx, ld, lrhs = reduce_triples(*stamp_on_host(n.nodal.ComponentTable(typ, val, a, b, kcl=mn, be=0), 4), mn)
    L = sps.csr_matrix((dx, ix, ip), shape=(nr, nr))[:mn, :mn].tocsr()
    L.sort_indices()
    assert np.array_equal(L.indptr, li) and np.array_equal(L.indices, lx) and L.data.tobytes() == ld.tobytes()
    assert rhs[:mn].tobytes() == lrhs.tobytes()
    assert host.collapsed(table, f) == mirror.collapsed(table, f) == 0


def test_amplifier_grid_ideal_pads_solves(tmp_path):
    table = case_table("amp_ideal", tmp_path)
    G, A = full_csr(table)
    x, parts = mirror.solve(table, G, A)
    want = sps.linalg.spsolve(G.tocsc(), A)
    assert block_err(x, want, table.kcl) <= 1e-9


def test_eligibility_rules(tmp_path):
    base = DOC["opmodel_amplifier.csv"]["rows"]
    assert mirror.reason(table_of(base, tmp_path)) == ""
    neg = table_of(base + [["rn", "R", "-2", "2", "g"]], tmp_path)
    assert mirror.reason(neg) == "not positive" and "not positive" in source_schur.skip_reason(neg)
    loop = table_of(HAND_TREE + [["vf", "E", "1", "1", "g"], ["vg", "E", "1", "2", "g"]], tmp_path)
    assert mirror.reason(loop) == "forest"
    # a VCVS whose two output leads are tied by a source: its current is undetermined
    t = table_of(HAND_TREE + [["e2", "VCVS", "3", "1", "2", "3", "g"]], tmp_path)
    f = mirror.forest(t)
    assert mirror.reason(t) == "one source tree" and host.collapsed(t, f) == mirror.collapsed(t, f) == 1
    # nodes touched only by dependent outputs: no reduced resistor reaches them
    t1 = table_of(DOC["test_1.csv"]["rows"], tmp_path)
    assert mirror.reason(t1) == "does not reach ground"
    assert mirror.reason(table_of(HAND_TREE, tmp_path), max_branches=2) == "schur_max_branches"


def _circuit(table, **opts):
    mode = sources.check_option(opts, table)
    return SimpleNamespace(table=table, sparse=True, _dist=None, _eliminate=mode,
                           _schur=schur.check_option(opts, True, opts.get("distributed")))


def test_option_matrix(tmp_path):
    mixed = table_of(HAND_TREE, tmp_path)
    assert source_schur.applies(_circuit(mixed, schur=True, eliminate_sources=True))
    with pytest.raises(ValueError):                                  # True alone: as before
        sources.check_option({"eliminate_sources": True}, mixed)
    with pytest.raises(ValueError):
        sources.check_option({"eliminate_sources": True, "schur": False}, mixed)
    assert not source_schur.applies(_circuit(mixed, schur=True))     # "auto": the full-system Schur
    assert not source_schur.applies(_circuit(mixed, schur=True, eliminate_sources=False))
    # without E rows or without dependent rows the combination is not asked for
    assert not source_schur.applies(_circuit(table_of(DOC["x_vcvs_null_control.csv"]["rows"], tmp_path), schur=True,
                                             eliminate_sources=True))
    assert not source_schur.applies(_circuit(table_of(orc.grid2d_rows(3) + [["v", "E", "1", "0", "g"]], tmp_path),
                                             schur=True, eliminate_sources=True))
    with pytest.raises(NotImplementedError):
        schur.check_option({"schur": True, "eliminate_sources": True}, True, True)


def test_amplifier_grid_ideal_pads_matches_csv(tmp_path):
    net = gen.amplifier_grid(12, 5, seed=3, pitch=4, dependents=2, ideal_pads=True)
    t = net.table()
    rows = _csv_rows(net)
    ref = n.Netlist(write_csv(rows, tmp_path / "amp.csv"))
    rt = ref.table()
    for col in ("type", "value", "a", "b", "c", "d", "drv", "branch"):
        assert getattr(rt, col).tobytes() == getattr(t, col).tobytes(), col
    assert (rt.kcl, rt.be) == (t.kcl, t.be) == (144 + 3 * 5 + 2 * 2, 9 + 5 + 3 * 2)
    assert dict(ref.nodenum) == {k: net.nodenum[k] for k in net.nodenum}
    assert ref.anomnum == dict(net.anomnum) and ref.ground == net.ground == "g"
    assert ref.table_and_currents()[1] == net.table_and_currents()[1]
    assert list(ref.component_keys) == list(net.component_keys)
    assert np.count_nonzero(t.type == K.T_A) == 144 and np.count_nonzero(t.type == K.T_E) == 9
    # the pads drop out of the Schur complement: 11 dependent rows instead of all 20 branch rows
    assert mirror.reason(t) == ""
    _, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    x, parts = mirror.solve(t, G.tocsr(), np.asarray(A, float))
    assert parts["md"] == 5 + 3 * 2 and block_err(x, want, t.kcl) <= 1e-9


def test_amplifier_grid_default_unchanged():
    """ideal_pads=False is the generator as before (pinned by its table bytes)."""
    import hashlib
    t = gen.amplifier_grid(12, 5, seed=3, pitch=4, dependents=2).table()
    h = hashlib.sha256()
    for col in ("type", "value", "a", "b", "c", "d", "drv", "branch"):
        h.update(getattr(t, col).tobytes())
    assert h.hexdigest() == "d2d0bda19f4d87c3ed91582a669f3c210df1dd8a55fe9f1474b1cacf30466f35"


def test_cli_mapping():
    from nodal_b200.cli import circuit_options, make_parser
    p = make_parser("t", "f")
    assert circuit_options(p.parse_args(["x.csv", "-s", "--schur", "--eliminate-sources", "on"])) == \
        {"eliminate_sources": True, "schur": True}
    assert circuit_options(p.parse_args(["x.csv", "-s", "--schur"])) == {"schur": True}
    assert "--schur" in p.format_help().split("--eliminate-sources")[1]
