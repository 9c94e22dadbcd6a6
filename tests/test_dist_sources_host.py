"""CPU statement of the row-partitioned elimination of the voltage sources (nodal_b200/dist_sources.py)
with the numpy statement of sources_mirror.py, for several world sizes: the E rows compacted per share,
the reduced shares, the rows each rank stamps (full and reduced), and the tree rows the expansion
gathers.  Shares of the table hold components [M r / R, M (r + 1) / R); several of them select nothing."""
import numpy as np
import pytest
import scipy.sparse as sps

import sources_mirror as mirror
from helpers import reduce_triples, stamp_on_host, write_csv
from test_sources_host import CASES, case_rows
import nodal_b200 as n
from nodal_b200 import dist as ndist
from nodal_b200 import generators as gen
from nodal_b200.device import coo_stride
from nodal_b200.table import ComponentTable

WORLDS = (1, 2, 3, 5, 8)


def share_bounds(table, world):
    m = len(table)
    return [(m * r // world, m * (r + 1) // world) for r in range(world)]


def subtable(table, idx):
    cols = [getattr(table, k)[idx] for k in ("type", "value", "a", "b", "c", "d", "drv", "branch")]
    return ComponentTable(*cols, kcl=table.kcl, be=table.be)


def mna_pick(t, rb, re):
    """The selection of nodal_table_select_mna_*: a lead in [rb, re), or an E row whose branch row is."""
    lead = ((t.a >= rb) & (t.a < re)) | ((t.b >= rb) & (t.b < re))
    br = t.kcl + t.branch
    return lead | ((t.type == mirror.T_E) & (br >= rb) & (br < re))


def lead_pick(t, rb, re):
    return ((t.a >= rb) & (t.a < re)) | ((t.b >= rb) & (t.b < re))


def exchange(shares, bounds, pick):
    """What every rank d receives: per source share (rank order) the selected components, share order kept.
    Returns per d the list of per-source index arrays (into the share)."""
    world = len(bounds) - 1
    return [[np.flatnonzero(pick(s, int(bounds[d]), int(bounds[d + 1]))) for s in shares] for d in range(world)]


def rows_of_csr(ip, ix, dt, rhs, rb, re):
    return ip[rb: re + 1] - ip[rb], ix[ip[rb]: ip[re]], dt[ip[rb]: ip[re]], rhs[rb:re]


def assert_rows_equal(got, want):
    for g, w in zip(got, want):
        assert np.ascontiguousarray(g).tobytes() == np.ascontiguousarray(w).tobytes()


def tables(tmp_path):
    out = {case: n.Netlist(write_csv(case_rows(case), tmp_path / f"{case}.csv")).table() for case in CASES}
    out["power_grid(64, 8)"] = gen.power_grid(64, 8, vdd=1.0, load=1e-3, seed=3).table()
    return out


@pytest.fixture(scope="module")
def all_tables(tmp_path_factory):
    return tables(tmp_path_factory.mktemp("dist_sources"))


@pytest.mark.parametrize("name", CASES + ["power_grid(64, 8)"])
@pytest.mark.parametrize("world", WORLDS)
def test_partitioned_statement(name, world, all_tables):
    table = all_tables[name]
    kcl, N = table.kcl, table.n
    f = mirror.forest(table)
    assert f["ok"]
    sb = share_bounds(table, world)
    shares = [subtable(table, np.arange(lo, hi)) for lo, hi in sb]

    # the E rows compacted per share, concatenated in rank order, are the table's E rows in order
    e_rows = [lo + np.flatnonzero(s.type == mirror.T_E) for (lo, _), s in zip(sb, shares)]
    assert np.array_equal(np.concatenate(e_rows), np.flatnonzero(table.type == mirror.T_E))

    # the reduced shares concatenated are the single-GPU reduced table, byte for byte
    parts = [mirror.reduce_table(s, f) for s in shares]
    want = mirror.reduce_table(table, f)
    for k in range(4):
        assert np.concatenate([p[k] for p in parts]).tobytes() == np.ascontiguousarray(want[k]).tobytes()

    # every rank's rows of the full MNA matrix from the components it receives
    stride = coo_stride(table)
    whole = reduce_triples(*stamp_on_host(table, stride), N)
    bounds = ndist.partition_rows(N, world)
    for d, picked in enumerate(exchange(shares, bounds, mna_pick)):
        idx = np.concatenate([lo + p for (lo, _), p in zip(sb, picked)])
        assert np.all(np.diff(idx) > 0)                          # global stamping order
        local = reduce_triples(*stamp_on_host(subtable(table, idx), stride), N)
        rb, re = int(bounds[d]), int(bounds[d + 1])
        assert_rows_equal(rows_of_csr(*local, rb, re), rows_of_csr(*whole, rb, re))

    # every rank's rows of the reduced system from the reduced shares (lead selection, m rows)
    m = f["rows"]
    rtab = [ComponentTable(*p, kcl=m, be=0) for p in parts]
    rwhole = reduce_triples(*stamp_on_host(ComponentTable(*want, kcl=m, be=0), 4), m)
    rbounds = ndist.partition_rows(m, world)
    for d, picked in enumerate(exchange(rtab, rbounds, lead_pick)):
        cols = [np.concatenate([p[k][sel] for p, sel in zip(parts, picked)]) for k in range(4)]
        local = reduce_triples(*stamp_on_host(ComponentTable(*cols, kcl=m, be=0), 4), m)
        rb, re = int(rbounds[d]), int(rbounds[d + 1])
        assert_rows_equal(rows_of_csr(*local, rb, re), rows_of_csr(*rwhole, rb, re))

    # the tree rows every rank contributes (its rows whose node has depth >= 1) carry all the expansion
    # reads: the currents from them alone equal the statement's from the whole residual
    ip, ix, dt, rhs = whole
    G = sps.csr_matrix((dt, ix, ip), shape=(N, N))
    y = np.random.default_rng(world).standard_normal(max(1, m))[:m]
    e = np.r_[mirror.potentials(f, y, kcl), np.zeros(N - kcl)]
    gx = G @ e
    depth = f["depth_of"]
    gathered = []
    for d in range(world):
        rb, re = int(bounds[d]), min(int(bounds[d + 1]), kcl)
        mine = np.arange(rb, max(rb, re))
        gathered.append(mine[depth[mine] >= 1])
    tree = np.concatenate(gathered)
    assert np.array_equal(tree, np.flatnonzero(depth[:kcl] >= 1))
    rho = np.full(kcl, np.nan)
    rho[tree] = rhs[tree] - gx[tree]
    got = mirror.expand(table, f, y, rho)
    assert got.tobytes() == mirror.expand(table, f, y, rhs[:kcl] - gx[:kcl]).tobytes()


def test_shares_that_select_nothing_are_covered(all_tables):
    """The cases above include shares without an E row and shares that send a rank nothing."""
    no_e = no_rows = 0
    for table in all_tables.values():
        for world in WORLDS:
            shares = [subtable(table, np.arange(lo, hi)) for lo, hi in share_bounds(table, world)]
            no_e += sum(not np.any(s.type == mirror.T_E) for s in shares)
            bounds = ndist.partition_rows(table.n, world)
            no_rows += sum(len(p) == 0 for picked in exchange(shares, bounds, mna_pick) for p in picked)
    assert no_e > 0 and no_rows > 0
