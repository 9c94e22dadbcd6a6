"""CPU checks of the voltage-source elimination: the numpy statement (sources_mirror.py) against the
oracle, csrc/sources_core.cuh compiled for the host against the statement bit for bit, the
eligibility rules, the power_grid generator and the CLI flag."""
import ctypes as C

import numpy as np
import pytest

import sources_mirror as mirror
from helpers import block_err, write_csv
from sources_host import sources_host_lib
import nodal_b200 as n
from nodal_b200 import constants as K
from nodal_b200 import generators as gen
from nodal_b200 import sources
from nodal_b200.options import parse
from oracle import mna_oracle as orc


def grid_rows(N, seed=0, load_prob=0.3):
    rng = np.random.default_rng(seed)
    rows = orc.grid2d_rows(N)
    nm = lambda x, y: "1" if (x, y) == (N // 2, N // 2) else "g" if (x, y) == (N // 2 + 2, N // 2 + 1) else f"n{x}_{y}"  # noqa: E731
    for x in range(N):
        for y in range(N):
            if rng.random() < load_prob and nm(x, y) != "g":
                rows.append([f"l{x}_{y}", "A", repr(float(rng.uniform(1e-4, 1e-3))), "g", nm(x, y)])
    return rows, nm


def case_rows(case):
    N = 12
    rows, nm = grid_rows(N, seed=CASES.index(case))
    if case in ("pads", "mixed"):
        k = 0
        for x in range(0, N, 4):
            for y in range(0, N, 4):
                if nm(x, y) not in ("g", "1"):
                    rows.append([f"v{k}", "E", "1.0", nm(x, y), "g"]); k += 1
    if case in ("floating", "mixed"):
        rows.append(["vf", "E", "0.25", nm(N - 2, N - 3), nm(N - 3, N - 3)])
    if case in ("chain", "mixed"):
        rows.append(["vs1", "E", "0.1", nm(1, N - 1), nm(2, N - 1)])
        rows.append(["vs2", "E", "0.2", nm(2, N - 1), nm(3, N - 1)])
        rows.append(["vs3", "E", "-0.3", nm(3, N - 1), "g"])
    if case == "bridge":           # two floating sources joined by a third: one floating tree of three
        rows.append(["va", "E", "0.5", nm(2, 2), nm(2, 3)])
        rows.append(["vb", "E", "0.7", nm(5, 5), nm(5, 6)])
        rows.append(["vab", "E", "0.3", nm(2, 3), nm(5, 5)])
    if case == "near_ground":      # anode on ground, and a source hanging off a node next to ground
        rows.append(["vg", "E", "0.4", "g", nm(N // 2 + 2, N // 2)])
        rows.append(["vn", "E", "0.2", nm(N // 2 + 2, N // 2 + 2), nm(N // 2 + 3, N // 2 + 1)])
    return rows


CASES = ["pads", "floating", "chain", "bridge", "near_ground", "mixed"]


def table_of(rows, tmp_path):
    return n.Netlist(write_csv(rows, tmp_path / "net.csv")).table()


@pytest.mark.parametrize("case", CASES)
def test_statement_matches_oracle(case, tmp_path):
    rows = case_rows(case)
    table = table_of(rows, tmp_path)
    onet, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    x, f = mirror.solve(table, G.tocsr(), A)
    assert f["loops"] == 0 and f["sources"] == table.be
    kcl = table.kcl
    assert block_err(x, want, kcl) <= 1e-12
    assert np.linalg.norm(G @ x - A) <= 1e-12 * np.linalg.norm(A)
    # the reduced matrix is the stamp of an R / A table: symmetric, one row per free tree
    Gr, _ = mirror.laplacian(*mirror.reduce_table(table, f), f["rows"])
    assert abs(Gr - Gr.T).max() == 0.0


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("case", CASES)
def test_core_matches_statement_bit_for_bit(case, tmp_path):
    rows = case_rows(case)
    table = table_of(rows, tmp_path)
    lib = sources_host_lib()
    f = mirror.forest(table)
    assert f["ok"]
    kcl = table.kcl
    depth = f["depth_of"]
    order = np.argsort(np.where(depth < 0, 1 << 30, depth), kind="stable").astype(np.int32)
    off = np.full(kcl + 1, np.nan)
    lib.src_offsets_host(kcl + 1, _p(order), _p(f["parent_edge"]), _p(table.value), _p(table.a), _p(table.b), kcl,
                         _p(off))
    assert off.tobytes() == f["offset"].tobytes()

    m = len(table)
    ot, ov = np.zeros(2 * m, np.uint8), np.zeros(2 * m)
    oa, ob = np.zeros(2 * m, np.int32), np.zeros(2 * m, np.int32)
    cnt = lib.src_reduce_table_host(m, _p(table.type), _p(table.value), _p(table.a), _p(table.b), kcl,
                                    _p(f["rep_row"]), _p(f["offset"]), _p(ot), _p(ov), _p(oa), _p(ob))
    want = mirror.reduce_table(table, f)
    assert cnt == len(want[0])
    for got, w in zip((ot, ov, oa, ob), want):
        assert got[:cnt].tobytes() == np.ascontiguousarray(w).tobytes()

    rng = np.random.default_rng(3)
    y = rng.standard_normal(max(1, f["rows"]))
    rho = rng.standard_normal(kcl)
    want = mirror.expand(table, f, y, rho)
    x = np.zeros(table.n)
    lib.src_expand_host(kcl, table.n, _p(f["rep_row"]), _p(f["offset"]), _p(f["parent_edge"]), _p(depth), f["depth"],
                        _p(table.a), _p(table.b), _p(table.branch), _p(y), _p(rho.copy()), _p(x))
    assert x.tobytes() == want.tobytes()


@pytest.mark.parametrize("extra, loops", [
    ([["vx", "E", "1", "n0_0", "g"], ["vy", "E", "2", "n0_0", "g"]], 1),                       # parallel sources
    ([["vx", "E", "1", "n0_0", "n0_1"], ["vy", "E", "1", "n0_1", "n1_1"],
      ["vz", "E", "1", "n1_1", "n0_0"]], 1),                                                 # a loop of three
    ([["vx", "E", "1", "n0_0", "n0_0"]], 1),                                                 # both leads on one node
    ([["vx", "E", "1", "g", "g"]], 1),                                                       # both leads on ground
])
def test_not_a_forest(extra, loops, tmp_path):
    rows = orc.grid2d_rows(6) + extra
    f = mirror.forest(table_of(rows, tmp_path))
    assert not f["ok"] and f["loops"] == loops


def test_shared_branch_is_not_eliminated(tmp_path):
    rows = orc.grid2d_rows(6) + [["v1", "E", "1", "n0_0", "g"], ["v1", "E", "1", "n3_3", "g"]]
    table = table_of(rows, tmp_path)
    assert table.be == 2 and list(table.branch[table.type == K.T_E]) == [1, 1]
    f = mirror.forest(table)
    assert not f["ok"] and f["branch_conflicts"] == 2


def test_eligibility_and_option_parsing(tmp_path):
    base = orc.grid2d_rows(6) + [["v1", "E", "1", "n0_0", "g"]]
    table = table_of(base, tmp_path)
    assert sources.skip_reason(table, "auto", 32768).startswith(f"{table.n} rows")
    assert sources.skip_reason(table, "auto", 10) == ""
    assert sources.skip_reason(table, True, 32768) == ""
    assert sources.skip_reason(table, False, 10) is None
    neg = table_of(base + [["rn", "R", "-2", "n1_1", "g"]], tmp_path)
    assert "not positive" in sources.skip_reason(neg, True, 32768)
    dep = table_of(base + [["d1", "VCVS", "2", "n5_5", "g", "n0_0", "g"]], tmp_path)
    assert sources.skip_reason(dep, "auto", 10) is None
    with pytest.raises(ValueError):
        parse({"eliminate_sources": True}, True, dep)
    assert parse({"eliminate_sources": "auto"}, True, dep).eliminate_sources == "auto"
    with pytest.raises(ValueError):
        parse({"eliminate_sources": "yes"}, True, table)
    assert sources.skip_reason(table_of(orc.grid2d_rows(6), tmp_path), True, 0) is None    # no E rows


def test_power_grid_matches_csv(tmp_path):
    net = gen.power_grid(10, 3, vdd=1.2, load=1e-3, seed=4)
    t = net.table()
    nodes = list(net.nodenum) + ["g"]
    name_of = lambda i: "g" if i < 0 else nodes[i]                       # noqa: E731
    keys = net.component_keys
    rows = [[keys[k], K.TYPE_NAME[int(t.type[k])], repr(float(t.value[k])), name_of(t.a[k]), name_of(t.b[k])]
            for k in range(len(t))]
    ref = n.Netlist(write_csv(rows, tmp_path / "pg.csv"))
    rt = ref.table()
    for col in ("type", "value", "a", "b", "branch"):
        assert getattr(rt, col).tobytes() == getattr(t, col).tobytes(), col
    assert (rt.kcl, rt.be) == (t.kcl, t.be) == (100, 16)
    assert dict(ref.nodenum) == {k: net.nodenum[k] for k in net.nodenum}
    assert ref.anomnum == dict(net.anomnum) and ref.ground == net.ground == "g"
    assert ref.table_and_currents()[1] == net.table_and_currents()[1]
    # the statement solves it: every pad at vdd, every node at or below it
    onet, G, A, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    x, f = mirror.solve(t, G.tocsr(), A)
    assert block_err(x, want, t.kcl) <= 1e-12
    assert f["rows"] == 84 and f["grounded_nodes"] == 16 and np.all(x[:t.kcl] <= 1.2)


def test_cli_flag():
    from nodal_b200.cli import circuit_options, make_parser
    p = make_parser("t", "f")
    assert circuit_options(p.parse_args(["x.csv", "-s"])) == {}
    assert circuit_options(p.parse_args(["x.csv", "-s", "--eliminate-sources", "on"])) == {"eliminate_sources": True}
    assert circuit_options(p.parse_args(["x.csv", "-s", "--eliminate-sources", "off"])) == {"eliminate_sources": False}
    assert circuit_options(p.parse_args(["x.csv", "--eliminate-sources", "on"])) == {}
