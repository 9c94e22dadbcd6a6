"""CPU checks of how a sparse Circuit chooses its solve path (nodal_b200/options.py): the parsed options,
their validation (same exception types and messages as before they were parsed in one place) and the
ordered candidates of the single-GPU sparse solve with the reasons the host declines them for."""
import numpy as np
import pytest

from helpers import golden, write_csv
import nodal_b200 as n
from nodal_b200 import generators as gen
from nodal_b200.options import SolveOptions, parse, plan
from oracle import mna_oracle as orc

DOC = golden("doc_netlists.json")
# E rows and dependent rows (tests/test_source_schur_host.py)
MIXED = [["ve", "E", "0.5", "1", "2"], ["r1", "R", "2", "1", "g"], ["r2", "R", "3", "2", "3"],
         ["r3", "R", "5", "3", "g"], ["r4", "R", "7", "3", "4"], ["r5", "R", "11", "4", "g"],
         ["e1", "VCVS", "2", "2", "4", "1", "3"], ["f1", "CCCS", "0.25", "3", "g", "2", "3", "r2"],
         ["h1", "CCVS", "1.5", "5", "g", "2", "3", "r2"], ["r6", "R", "13", "5", "1"]]
KEPT = "the GMRES / dense-LU path is kept"


def table_of(rows, tmp_path):
    return n.Netlist(write_csv(rows, tmp_path / "net.csv")).table()


def steps(table, sparse=True, **options):
    return [(c.path, c.key, c.reason) for c in plan(table, parse(options, sparse, table))]


def test_plan_resistor_grid(tmp_path):
    table = gen.grid2d(12).table()
    assert steps(table) == []
    assert steps(table, eliminate_sources=True) == []
    (c,) = plan(table, parse({"schur": True}, True, table))
    assert (c.path, c.key, c.reason) == ("schur", "schur", "no branch rows")
    assert c.declined == dict(applied=False, branches=0, node_rows=table.kcl, reason="no branch rows")


def test_plan_sources_by_size():
    small = gen.power_grid(40, 8, vdd=1.0, load=1e-3, seed=1).table()
    assert small.n <= 32768
    reason = f"{small.n} rows <= dense_fallback_max_rows (32768): {KEPT}"
    (c,) = plan(small, parse({}, True, small))
    assert (c.path, c.key, c.reason, c.declined) == ("sources", "reduction", reason,
                                                     dict(eliminated=False, reason=reason))
    assert steps(small, eliminate_sources=True) == [("sources", "reduction", "")]
    assert steps(small, dense_fallback_max_rows=small.n) == [
        ("sources", "reduction", f"{small.n} rows <= dense_fallback_max_rows ({small.n}): {KEPT}")]
    assert steps(small, dense_fallback_max_rows=small.n - 1) == [("sources", "reduction", "")]
    assert steps(small, eliminate_sources=False) == []
    large = gen.power_grid(200, 16, vdd=1.0, load=1e-3, seed=1).table()
    assert large.n > 32768
    assert steps(large) == [("sources", "reduction", "")]
    assert steps(large, eliminate_sources=False) == []
    # an R / A / E table with schur=True: the elimination first, then the Schur complement
    assert steps(large, schur=True) == [("sources", "reduction", ""), ("schur", "schur", "")]
    assert steps(small, schur=True) == [("sources", "reduction", reason), ("schur", "schur", "")]


def test_plan_nonpositive_resistance(tmp_path):
    neg = table_of(orc.grid2d_rows(6) + [["v1", "E", "1", "n0_0", "g"], ["rn", "R", "-2", "n1_1", "g"]], tmp_path)
    assert steps(neg, eliminate_sources=True, schur=True) == [
        ("sources", "reduction", "a resistance is not positive (the reduced system would not be SPD)"),
        ("schur", "schur", "a resistance is not positive (L would not be SPD)")]
    mixed = table_of(MIXED + [["rn", "R", "-2", "2", "g"]], tmp_path)
    assert steps(mixed, eliminate_sources=True, schur=True) == [
        ("source_schur", "reduction", "a resistance is not positive (the reduced L would not be SPD)"),
        ("schur", "schur", "a resistance is not positive (L would not be SPD)")]
    (c, _) = plan(mixed, parse(dict(eliminate_sources=True, schur=True), True, mixed))
    assert c.declined == dict(eliminated=False, applied=False, reason=c.reason)


def test_plan_opamps(tmp_path):
    amp = table_of(DOC["opmodel_amplifier.csv"]["rows"], tmp_path)
    assert steps(amp) == []
    assert steps(amp, schur=True) == [("schur", "schur", "")]
    assert steps(amp, schur=True, schur_max_branches=amp.be - 1) == [
        ("schur", "schur", f"{amp.be} branch rows > schur_max_branches ({amp.be - 1})")]
    grid = gen.amplifier_grid(12, 5, seed=3, pitch=4, dependents=2).table()
    assert steps(grid) == [] and steps(grid, schur=True) == [("schur", "schur", "")]


def test_plan_ideal_pads():
    t = gen.amplifier_grid(12, 5, seed=3, pitch=4, dependents=2, ideal_pads=True).table()
    assert steps(t) == []
    assert steps(t, schur=True) == [("schur", "schur", "")]
    assert steps(t, schur=True, eliminate_sources=False) == [("schur", "schur", "")]
    assert steps(t, schur=True, eliminate_sources=True) == [("source_schur", "reduction", ""),
                                                           ("schur", "schur", "")]


@pytest.mark.parametrize("eliminate", ["auto", True, False])
@pytest.mark.parametrize("schur", [False, True])
@pytest.mark.parametrize("distributed", [False, True])
def test_eliminate_schur_distributed(eliminate, schur, distributed, tmp_path):
    """Every combination on a table with E and dependent rows, and on an R / A / E one."""
    mixed = table_of(MIXED, tmp_path)
    rae = gen.power_grid(40, 8, vdd=1.0, load=1e-3, seed=1).table()
    options = dict(eliminate_sources=eliminate, schur=schur, distributed=distributed)
    if schur and distributed:
        for table in (mixed, rae):
            with pytest.raises(NotImplementedError, match="runs on one GPU"):
                parse(options, True, table)
        return
    if eliminate is True and not schur and not distributed:
        with pytest.raises(ValueError, match="needs a netlist of R, A and E rows only"):
            parse(options, True, mixed)
    else:
        opts = parse(options, True, mixed)
        want = (["source_schur"] if schur and eliminate is True else []) + (["schur"] if schur else [])
        assert [c.path for c in plan(mixed, opts)] == want
    opts = parse(options, True, rae)
    want = ([] if eliminate is False else ["sources"]) + (["schur"] if schur else [])
    assert [c.path for c in plan(rae, opts)] == want


def _errors(tmp_path):
    """(options, sparse, table, exception, message) of every invalid option, the messages as they were."""
    mixed = table_of(MIXED, tmp_path)
    grid = gen.grid2d(6).table()
    return [
        (dict(schur="yes"), True, grid, ValueError, "schur must be True or False, got 'yes'"),
        (dict(schur=1), True, grid, ValueError, "schur must be True or False, got 1"),
        (dict(schur=None), False, grid, ValueError, "schur must be True or False, got None"),
        (dict(schur=True), False, grid, ValueError, "schur=True needs sparse=True (the dense path already solves by LU)"),
        (dict(schur=True, distributed=True), True, grid, NotImplementedError,
         "the Schur-complement solve runs on one GPU (distributed=True is not supported)"),
        (dict(schur_refine=-1), True, grid, ValueError, "schur_refine must be >= 0"),
        (dict(schur_refine=-1), False, grid, ValueError, "schur_refine must be >= 0"),
        (dict(schur_max_branches=0), True, grid, ValueError, "schur_max_branches must be >= 1"),
        (dict(eliminate_sources="yes"), True, grid, ValueError,
         "eliminate_sources must be 'auto', True or False, got 'yes'"),
        (dict(eliminate_sources=True), True, mixed, ValueError,
         "eliminate_sources=True needs a netlist of R, A and E rows only (dependent sources cannot be "
         "eliminated; with schur=True they go through the Schur complement of the reduced system)"),
        (dict(eliminate_sources=True, schur=False), True, mixed, ValueError,
         "eliminate_sources=True needs a netlist of R, A and E rows only (dependent sources cannot be "
         "eliminated; with schur=True they go through the Schur complement of the reduced system)"),
        (dict(precond="ilu"), True, grid, ValueError, "precond must be 'auto', 'jacobi' or 'amg', got 'ilu'"),
        (dict(x0=np.zeros(3)), True, grid, ValueError, f"x0 must have {grid.n} entries"),
        (dict(x0=np.zeros((grid.n, 1))), True, grid, ValueError, f"x0 must have {grid.n} entries"),
    ]


def test_invalid_options(tmp_path):
    for options, sparse, table, exc, message in _errors(tmp_path):
        with pytest.raises(exc) as info:
            parse(options, sparse, table)
        assert type(info.value) is exc and str(info.value) == message, (options, str(info.value))


def test_invalid_options_at_construction(tmp_path):
    """Circuit parses its options before it needs a device."""
    net = n.Netlist(write_csv(MIXED, tmp_path / "mixed.csv"))
    with pytest.raises(ValueError, match="needs sparse=True"):
        n.Circuit(net, sparse=False, schur=True)
    with pytest.raises(ValueError, match="R, A and E rows only"):
        n.Circuit(net, sparse=True, eliminate_sources=True)
    with pytest.raises(ValueError, match="precond must be"):
        n.Circuit(net, sparse=True, precond="ilu")


def test_checks_only_on_the_sparse_path():
    """precond, eliminate_sources and x0 are only read by the sparse path: a dense Circuit ignores them."""
    grid = gen.grid2d(6).table()
    opts = parse(dict(precond="ilu", x0=np.zeros(3), eliminate_sources="yes"), False, grid)
    assert opts.precond == "ilu" and opts.eliminate_sources == "yes"
    # x0 is not read by the row-partitioned solve
    assert parse(dict(x0=np.zeros(3), distributed=True), True, grid).distributed


def test_parsed_values():
    grid = gen.grid2d(6).table()
    opts = parse({"unknown_key": 1, "precond": "jacobi"}, True, grid)
    assert opts == SolveOptions(precond="jacobi")
    assert opts.spd_solver == "pcg" and parse({}, True, grid).spd_solver == "amg"
    assert parse({"precond": "amg"}, True, grid).spd_solver == "amg"
    # rtol not given: 1e-10, GMRES 1e-12, the L solves of the Schur paths rtol
    assert (opts.spd_rtol, opts.gmres_rtol, opts.inner_rtol) == (1e-10, 1e-12, 1e-10)
    given = parse(dict(rtol=1e-8), True, grid)
    assert (given.spd_rtol, given.gmres_rtol, given.inner_rtol) == (1e-8, 1e-8, 1e-8)
    assert parse(dict(rtol=1e-8, schur_rtol=1e-9), True, grid).inner_rtol == 1e-9
    assert (opts.gmres_maxit, parse(dict(maxit=7), True, grid).gmres_maxit) == (20000, 7)
    assert opts.amg_params == {} and parse(dict(amg={"coarse": 64}), True, grid).amg_params == {"coarse": 64}
    assert parse(dict(schur_refine="3", dense_fallback_max_rows=1e5), True, grid).schur_refine == 3
    x0 = parse(dict(x0=list(range(grid.n))), True, grid).x0
    assert x0.dtype == np.float64 and x0.flags.c_contiguous and x0.shape == (grid.n,)
