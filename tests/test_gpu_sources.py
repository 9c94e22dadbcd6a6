"""The voltage-source elimination on the device (csrc/sources.cu): forest and reduced table bit for
bit against the numpy statement, the reduced CSR against the CSR model, solutions against the
oracle, the 4096^2 power grid's properties, the fall-backs and reproducibility."""
import warnings

import numpy as np
import pytest

import sources_mirror as mirror
from helpers import block_err, reduce_triples, stamp_on_host, write_csv
from test_sources_host import CASES, case_rows
import nodal_b200 as n
from nodal_b200 import constants as K
from nodal_b200 import generators as gen
from nodal_b200.device import Device
from oracle import mna_oracle as orc

pytestmark = pytest.mark.gpu


def netlist(rows, tmp_path, name="net.csv"):
    return n.Netlist(write_csv(rows, tmp_path / name))


def rows_of(net):
    """csv rows of a generated netlist (names as the csv path numbers them)."""
    t = net.table()
    nodes = list(net.nodenum) + [net.ground]
    keys = net.component_keys
    return [[keys[k], K.TYPE_NAME[int(t.type[k])], repr(float(t.value[k])), nodes[t.a[k]], nodes[t.b[k]]]
            for k in range(len(t))]


def device_forest(table):
    dev = Device.get(0)
    dtab = dev.upload_table(table)
    info, f = dev.source_forest(dtab, len(table), table.kcl, table.be)
    return dev, dtab, info, f


@pytest.mark.parametrize("case", CASES)
def test_forest_and_reduced_table_match_statement(case, tmp_path):
    table = netlist(case_rows(case), tmp_path).table()
    dev, dtab, info, f = device_forest(table)
    want = mirror.forest(table)
    for k in ("sources", "loops", "branch_conflicts", "trees", "floating_trees", "grounded_nodes", "rows", "depth"):
        assert info[k] == want[k], k
    kcl = table.kcl
    for k, w in (("rep_row", "rep_row"), ("offset", "offset"), ("parent_edge", "parent_edge"), ("depth", "depth_of")):
        assert f[k].cpu().numpy().tobytes() == want[w].tobytes(), k
    assert f["roots"][: info["rows"]].cpu().numpy().tobytes() == want["roots"].tobytes()
    red, m = dev.source_reduce(dtab, len(table), kcl, f)
    wt, wv, wa, wb = mirror.reduce_table(table, want)
    assert m == len(wt)
    got = [red[k][:m].cpu().numpy() for k in ("type", "value", "a", "b")]
    for g, w in zip(got, (wt, wv, wa, wb)):
        assert g.tobytes() == np.ascontiguousarray(w).tobytes()
    # the reduced CSR is the CSR model of that table
    rt = n.ComponentTable(*got, kcl=info["rows"], be=0)
    csr, rhs = dev.assemble_csr_raw(red, m, info["rows"], info["rows"], 4)
    ip, ix, dv, rb = reduce_triples(*stamp_on_host(rt, 4), rt.n)
    assert csr.indptr.cpu().numpy().tobytes() == ip.tobytes()
    assert csr.indices.cpu().numpy().tobytes() == ix.tobytes()
    assert csr.data.cpu().numpy().tobytes() == dv.tobytes()
    assert rhs.cpu().numpy().tobytes() == rb.tobytes()


@pytest.mark.parametrize("case", CASES)
def test_eliminated_solve_matches_oracle(case, tmp_path):
    rows = case_rows(case)
    _, _, _, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    net = netlist(rows, tmp_path)
    sol = n.Circuit(net, sparse=True, eliminate_sources=True).solve()
    red = sol.stats["reduction"]
    assert red["eliminated"] and red["relres_full"] <= 1e-9
    kcl = net.nums["kcl"]
    assert block_err(sol.result[:kcl], want[:kcl], kcl) <= 1e-9
    assert block_err(sol.result[kcl:], want[kcl:], 0) <= 1e-9


def test_auto_route_on_200_grid_matches_oracle():
    net = gen.power_grid(200, 16, vdd=1.0, load=1e-3, seed=1)
    assert net.table().n > 32768
    # the currents are differences of KCL residuals: 1e-10 on the reduced solve leaves them ~1e-9 off
    sol = n.Circuit(net, sparse=True, rtol=1e-12).solve()
    red = sol.stats["reduction"]
    assert red["eliminated"] and red["relres_full"] <= 1e-9 and sol.stats["status"] == 0
    _, _, _, _, want = orc.solve_rows(rows_of(net), sparse=True, backend="dict")
    kcl = net.nums["kcl"]
    assert block_err(sol.result[:kcl], want[:kcl], kcl) <= 1e-9
    assert block_err(sol.result[kcl:], want[kcl:], 0) <= 1e-9
    # the same netlist below the size limit keeps the existing path
    small = n.Circuit(net, sparse=True, dense_fallback_max_rows=10**6)
    assert small._dtab is None


def test_power_grid_4096():
    N, vdd = 4096, 1.0
    net = gen.power_grid(N, 64, vdd=vdd, load=1e-4, seed=0)
    table = net.table()
    circuit = n.Circuit(net, sparse=True)
    sol = circuit.solve()
    st, red = sol.stats, sol.stats["reduction"]
    assert st["status"] == 0 and red["eliminated"] and red["relres_full"] <= 1e-9
    assert red["sources"] == 64 * 64 and red["reduced_rows"] == N * N - 64 * 64 and red["forest_depth"] == 1
    x = sol.result
    assert np.all(np.isfinite(x))
    load = float(table.value[table.type == K.T_A].sum())
    assert abs(float(x[table.kcl:].sum()) - load) <= 1e-9 * load
    assert np.all(x[: table.kcl] <= vdd)
    # residual re-checked with the CSR SpMV of the library, norms on the host
    dev = Device.get(0)
    gx = dev.spmv(circuit.G, dev.to_device(x)).cpu().numpy()
    A = circuit.A_host
    assert np.linalg.norm(A - gx) <= 1e-9 * np.linalg.norm(A)


def test_loop_with_true_is_the_existing_path(tmp_path):
    rows = case_rows("pads") + [["vp", "E", "1.0", "n0_0", "g"]]        # parallel to pad v0
    net = netlist(rows, tmp_path)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        on = n.Circuit(net, sparse=True, eliminate_sources=True).solve()
        off = n.Circuit(net, sparse=True, eliminate_sources=False).solve()
    red = on.stats.pop("reduction")
    assert not red["eliminated"] and "forest" in red["reason"]
    assert "reduction" not in off.stats
    assert on.stats == off.stats
    assert np.array_equal(on.result, off.result, equal_nan=True)


def test_check_connected_still_raises(tmp_path):
    rows = case_rows("pads") + [["rf", "R", "1", "f1", "f2"]]
    net = netlist(rows, tmp_path)
    with pytest.raises(n.UnconnectedCircuitError):
        n.Circuit(net, sparse=True, eliminate_sources=True, check_connected=True).solve()


def test_runs_are_bitwise_equal_and_x0_is_accepted():
    net = gen.power_grid(300, 20, vdd=1.0, load=1e-3, seed=2)
    a = n.Circuit(net, sparse=True).solve()
    b = n.Circuit(net, sparse=True).solve()
    assert a.stats["reduction"]["eliminated"]
    assert a.result.tobytes() == b.result.tobytes()
    warm = n.Circuit(net, sparse=True, x0=a.result).solve()
    assert warm.stats["reduction"]["eliminated"] and warm.stats["status"] == 0
    assert warm.stats["iterations"] <= a.stats["iterations"]
    assert block_err(warm.result, a.result, net.nums["kcl"]) <= 1e-9
    with pytest.raises(ValueError):
        n.Circuit(net, sparse=True, x0=np.zeros(3)).solve()
