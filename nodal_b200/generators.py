"""Synthetic netlists of BASELINE.json's configs, produced directly as component tables.

At C5 sizes (33.5 M resistors) the reference's ingest -- csv parsing into a dict of
Component objects, then a deepcopy in equivalent_resistance -- takes tens of minutes, so
the benchmarks feed the struct-of-arrays table directly (SURVEY.md section 7.3 item 7).
``TableNetlist`` is a Netlist whose storage *is* the table; its numbering is computed
with vectorised numpy following exactly the reference's first-appearance rule
(nodal/nodal.py:249-257,283-287), which tests check against the csv path.
"""
from __future__ import annotations

import copy
from collections.abc import Mapping

import numpy as np

from . import constants as K
from .nodal import Netlist
from .table import ComponentTable


def first_appearance_numbering(a_id, b_id, ground_id):
    """Row index of every node id under the reference's rule: walk components in
    order, leads in (anode, bnode) order, number nodes at first sight, skip ground.

    a_id, b_id: int arrays of arbitrary non-negative node ids.  Returns
    (index_of_id: dict-like array sized max_id+1 with -1 for ground, kcl)."""
    inter = np.empty(2 * len(a_id), dtype=np.int64)
    inter[0::2] = a_id
    inter[1::2] = b_id
    size = int(inter.max()) + 1
    first = np.full(size, np.iinfo(np.int64).max, dtype=np.int64)
    # repeated fancy-index assignment keeps the LAST write; walking backwards makes that
    # the first appearance
    first[inter[::-1]] = np.arange(len(inter) - 1, -1, -1, dtype=np.int64)
    present = np.flatnonzero(first != np.iinfo(np.int64).max)
    order = present[np.argsort(first[present], kind="stable")]   # node ids in discovery order
    order = order[order != ground_id]
    index = np.full(size, -1, dtype=np.int32)
    index[order] = np.arange(len(order), dtype=np.int32)
    return index, len(order)


class _LazyNodeMap(Mapping):
    """nodenum of a generated netlist: name -> row index without materialising
    millions of strings.  `encode(name) -> node id or None`, `decode(id) -> name`."""

    def __init__(self, index, encode, decode, kcl):
        self._index, self._encode, self._decode, self._kcl = index, encode, decode, kcl

    def __getitem__(self, name):
        nid = self._encode(name)
        if nid is None or nid >= len(self._index) or self._index[nid] < 0:
            raise KeyError(name)
        return int(self._index[nid])

    def __contains__(self, name):
        nid = self._encode(name)
        return nid is not None and 0 <= nid < len(self._index) and self._index[nid] >= 0

    def __len__(self):
        return self._kcl

    def __iter__(self):
        order = np.argsort(np.where(self._index >= 0, self._index, np.iinfo(np.int32).max),
                           kind="stable")[: self._kcl]
        for nid in order:
            yield self._decode(int(nid))


class TableNetlist(Netlist):
    """Netlist backed by a ComponentTable (no per-component Python objects)."""

    def __init__(self, table, nodenum, ground, names=None, anomnum=None, node_ids=None):
        # deliberately does not call Netlist.__init__ (no file to read)
        self._table = table
        self.nodenum = nodenum
        self.ground = ground
        self.anomnum = anomnum or {}
        self.nums = {"components": len(table), "anomalies": table.be, "be": table.be,
                     "kcl": table.kcl, "opamps": 0}
        self._names = names           # optional callable k -> component name
        self.opmodel_equivalents = []
        self._currents = []

    # dict-of-Component views are not materialised for generated netlists
    @property
    def components(self):
        raise AttributeError("TableNetlist keeps components as a struct-of-arrays table; "
                             "use .table()")

    @property
    def component_keys(self):
        if getattr(self, "_component_names", None) is not None:      # Arrow column kept by the ingest
            from .ingest import _pylist
            return _pylist(self._component_names)
        f = self._names or (lambda k: f"c{k}")
        return [f(k) for k in range(len(self._table))]

    @property
    def degrees(self):
        if getattr(self, "_degrees", None) is not None:
            return self._degrees
        raise AttributeError("this TableNetlist does not keep per-node degrees")

    def is_resistive(self):
        return self._table.is_resistive()

    def table_and_currents(self):
        return self._table, list(self._currents)

    def table(self):
        return self._table

    def process_component(self, data):
        """Late registration of one more component between EXISTING nodes (what
        equivalent_resistance does, equiv.py:51).  Only R and A rows are supported."""
        if data == [] or data[0][0] == "#":
            return
        kind = data[K.TCOL]
        if kind not in ("R", "A"):
            raise NotImplementedError("TableNetlist.process_component supports R and A rows")
        idx = [K.GROUND if node == self.ground else self.nodenum[node]
               for node in (data[K.ACOL], data[K.BCOL])]
        self._table = self._table.append(K.TYPE_CODE[kind], float(data[K.VCOL]), idx[0], idx[1])
        self.nums["components"] += 1

    def __deepcopy__(self, memo):
        dup = copy.copy(self)          # the table is immutable from our side: append() copies
        dup.nums = dict(self.nums)
        dup._currents = list(self._currents)
        return dup


# --------------------------------------------------------------------------- resistor lattices
def _lattice(shape, probe, ground_pos, resistance):
    """Resistor lattice of arbitrary dimension, generator loop order of SURVEY.md 8(d):
    for every site in row-major order of `shape`, one resistor to the +1 neighbour along
    each axis in turn."""
    shape = tuple(int(s) for s in shape)
    nd = len(shape)
    sites = int(np.prod(shape))
    strides = [int(np.prod(shape[k + 1:])) for k in range(nd)]
    sid = np.arange(sites, dtype=np.int64)
    coords = np.unravel_index(sid, shape)
    # per site, per axis: does the +1 neighbour exist?  emission order = site major, axis minor
    has = np.stack([coords[k] + 1 < shape[k] for k in range(nd)], axis=1)      # (sites, nd)
    nb = np.stack([sid + strides[k] for k in range(nd)], axis=1)
    a_id = np.repeat(sid, nd).reshape(sites, nd)[has]
    b_id = nb[has]
    gid = int(np.ravel_multi_index(ground_pos, shape))
    pid = int(np.ravel_multi_index(probe, shape))
    index, kcl = first_appearance_numbering(a_id, b_id, gid)
    a = index[a_id]
    b = index[b_id]
    m = len(a)
    table = ComponentTable(np.full(m, K.T_R, np.uint8), np.full(m, float(resistance)), a, b,
                           kcl=kcl, be=0)

    def encode(name):
        if name == "1":
            return pid
        if name == "g":
            return gid
        if not name.startswith("n"):
            return None
        try:
            pos = tuple(int(t) for t in name[1:].split("_"))
        except ValueError:
            return None
        if len(pos) != nd or any(not (0 <= p < s) for p, s in zip(pos, shape)):
            return None
        nid = int(np.ravel_multi_index(pos, shape))
        return None if nid in (pid, gid) else nid      # those two are only known as "1" / "g"

    def decode(nid):
        if nid == pid:
            return "1"
        if nid == gid:
            return "g"
        return "n" + "_".join(str(int(v)) for v in np.unravel_index(nid, shape))

    nodenum = _LazyNodeMap(index, encode, decode, kcl)
    return TableNetlist(table, nodenum, "g", names=lambda k: f"r{k}")


def grid2d(N, resistance=1.0):
    """Config C2 / C5a: N x N grid of equal resistors; probe node "1" at (N//2, N//2),
    ground "g" a knight's move away at (N//2+2, N//2+1) (xkcd 356)."""
    return _lattice((N, N), (N // 2, N // 2), (N // 2 + 2, N // 2 + 1), resistance)


def lattice3d(N, resistance=1.0):
    """Config C5b: N^3 lattice, "1" at the centre, "g" at (N/2+2, N/2+1, N/2)."""
    h = N // 2
    return _lattice((N, N, N), (h, h, h), (h + 2, h + 1, h), resistance)


# --------------------------------------------------------------------------- power-delivery grid
def power_grid(N, pitch, vdd=1.0, load=1e-4, seed=0, resistance=1.0):
    """Resistive N x N mesh held by supply pads (IR-drop analysis): the resistors of grid2d's loop
    order between nodes "n{x}_{y}", then one E source "v{k}" of `vdd` from every node with x and y
    multiples of `pitch` to ground "g" (row-major), then a load "l{k}" on every node (row-major):
    an A row from "g" to the node drawing a current uniform in [0, load) (seed).  Numbering,
    anomnum and branch are those of the csv path (first appearance; branch k = pad k)."""
    N, pitch = int(N), int(pitch)
    if N < 2 or pitch < 1:
        raise ValueError("power_grid needs N >= 2 and pitch >= 1")
    rng = np.random.default_rng(seed)
    sites = N * N
    sid = np.arange(sites, dtype=np.int64)
    x, y = sid // N, sid % N
    has = np.stack([x + 1 < N, y + 1 < N], axis=1)
    nb = np.stack([sid + N, sid + 1], axis=1)
    ra = np.repeat(sid, 2).reshape(sites, 2)[has]
    rb = nb[has]
    gid = sites
    pads = sid[(x % pitch == 0) & (y % pitch == 0)]
    P = len(pads)
    a_id = np.concatenate([ra, pads, np.full(sites, gid)])
    b_id = np.concatenate([rb, np.full(P, gid), sid])
    index, kcl = first_appearance_numbering(a_id, b_id, gid)
    m_r = len(ra)
    type_ = np.concatenate([np.full(m_r, K.T_R, np.uint8), np.full(P, K.T_E, np.uint8), np.full(sites, K.T_A, np.uint8)])
    value = np.concatenate([np.full(m_r, float(resistance)), np.full(P, float(vdd)), rng.uniform(0.0, load, sites)])
    branch = np.full(len(type_), -1, np.int32)
    branch[m_r:m_r + P] = np.arange(P, dtype=np.int32)
    table = ComponentTable(type_, value, index[a_id], index[b_id], branch=branch, kcl=kcl, be=P)

    def encode(name):
        if name == "g":
            return gid
        if not name.startswith("n"):
            return None
        try:
            px, py = (int(t) for t in name[1:].split("_"))
        except ValueError:
            return None
        return px * N + py if 0 <= px < N and 0 <= py < N else None

    def decode(nid):
        return "g" if nid == gid else f"n{nid // N}_{nid % N}"

    def names(k):
        k = int(k)
        return f"r{k}" if k < m_r else f"v{k - m_r}" if k < m_r + P else f"l{k - m_r - P}"

    net = TableNetlist(table, _LazyNodeMap(index, encode, decode, kcl), "g", names=names,
                       anomnum=_PadNames(P))
    net._currents = [f"v{k}" for k in range(P)]
    return net


class _PadNames(Mapping):
    """anomnum of power_grid: "v{k}" -> k without materialising the names."""

    def __init__(self, count):
        self._count = count

    def __getitem__(self, name):
        if isinstance(name, str) and name.startswith("v") and name[1:].isdigit():
            k = int(name[1:])
            if k < self._count and name == f"v{k}":
                return k
        raise KeyError(name)

    def __len__(self):
        return self._count

    def __iter__(self):
        return (f"v{k}" for k in range(self._count))


# --------------------------------------------------------------------------- amplifiers on a sheet
def amplifier_grid(N, stages, seed=0, pitch=None, dependents=4, resistance=1.0, vdd=1.0, ideal_pads=False):
    """Op-amp stages coupled through a resistive N x N sheet (the workload of the Schur-complement
    solve, nodal_b200/schur.py): the resistors of grid2d's loop order between nodes "n{x}_{y}", a load
    resistor "l{k}" to ground "g" on every node (row-major), supply pads every `pitch` nodes (default
    N // 8) as an E source "v{k}" of `vdd` behind a series resistor "rs{k}" (node "s{k}"), then per stage
    p a non-inverting amplifier: OPMODEL "q{p}" reading a random sheet node, gain 1 + rf/rg <= 100
    ("rg{p}" to ground), driving another random sheet node through "rd{p}" from its output "o{p}";
    then `dependents` each of VCVS "dv{k}", CCVS "hv{k}" (driving "xv{k}" / "xh{k}", tied to the sheet
    by "rx{k}" / "rh{k}") and CCCS "fv{k}" (into a sheet node), the current-controlled ones driven by
    sheet resistors.  Every node reaches ground through resistors.  Component order, numbering,
    anomnum and branches are those of the csv path of the same rows (OPMODEL rows expand after all
    others, as ri, ro, vcvs, rf).

    ideal_pads=True: the sheet is held by ideal pads, as in power_grid -- every pad is an E source
    "v{k}" of `vdd` from its sheet node straight to ground (no "rs{k}" / "s{k}"), and the load "l{k}"
    on every node is an A row from ground drawing vdd / (the load resistance).  The sheet then reaches
    ground through the pads and, through resistors, only by way of the amplifier stages; every pad is a
    branch row (the workload of nodal_b200/source_schur.py)."""
    N, stages, dependents = int(N), int(stages), int(dependents)
    pitch = max(1, N // 8) if pitch is None else int(pitch)
    if N < 2 or stages < 0 or dependents < 0 or pitch < 1:
        raise ValueError("amplifier_grid needs N >= 2, stages >= 0, dependents >= 0 and pitch >= 1")
    rng = np.random.default_rng(seed)
    sites = N * N
    sid = np.arange(sites, dtype=np.int64)
    x, y = sid // N, sid % N
    has = np.stack([x + 1 < N, y + 1 < N], axis=1)
    nb = np.stack([sid + N, sid + 1], axis=1)
    ra = np.repeat(sid, 2).reshape(sites, 2)[has]
    rb = nb[has]
    m_r = len(ra)
    gid = sites
    extra_names = []                                   # node ids gid + 1, ... of the named nodes

    def node(name):
        extra_names.append(name)
        return gid + len(extra_names)

    pads = sid[(x % pitch == 0) & (y % pitch == 0)]
    # (name, type, value, a, b, c, d, driver row) of the rows after the sheet and the loads
    rows = []
    for k, p in enumerate(pads):
        if ideal_pads:
            rows.append((f"v{k}", K.T_E, float(vdd), int(p), gid, -1, -1, -1))
            continue
        s = node(f"s{k}")
        rows.append((f"rs{k}", K.T_R, float(10 ** rng.uniform(-2, -1)), s, int(p), -1, -1, -1))
        rows.append((f"v{k}", K.T_E, float(vdd), s, gid, -1, -1, -1))
    amp = []
    for p in range(stages):
        pos, drive = (int(v) for v in rng.integers(0, sites, size=2))
        out, neg = node(f"o{p}"), node(f"m{p}")
        rf = float(10 ** rng.uniform(2, 4))
        rg = rf / float(rng.uniform(0.5, 99.0))
        rows.append((f"rg{p}", K.T_R, rg, neg, gid, -1, -1, -1))
        rows.append((f"rd{p}", K.T_R, float(10 ** rng.uniform(0, 2)), out, drive, -1, -1, -1))
        amp.append((p, rf, out, pos, neg))
    for k in range(dependents):
        c1, c2, t1, t2, t3 = (int(v) for v in rng.integers(0, sites, size=5))
        dh, df = (int(v) for v in rng.integers(0, m_r, size=2))
        xv, xh = node(f"xv{k}"), node(f"xh{k}")
        rows.append((f"dv{k}", K.T_VCVS, float(rng.uniform(-2, 2)), xv, gid, c1, c2, -1))
        rows.append((f"rx{k}", K.T_R, float(10 ** rng.uniform(1, 3)), xv, t1, -1, -1, -1))
        rows.append((f"hv{k}", K.T_CCVS, float(rng.uniform(-2, 2)), xh, gid, int(ra[dh]), int(rb[dh]), dh))
        rows.append((f"rh{k}", K.T_R, float(10 ** rng.uniform(1, 3)), xh, t2, -1, -1, -1))
        rows.append((f"fv{k}", K.T_CCCS, float(rng.uniform(-0.5, 0.5)), t3, gid, int(ra[df]), int(rb[df]), df))
    for p, rf, out, pos, neg in amp:                   # the OPMODEL expansion (nodal.py build_opmodel)
        inner = node(f"q{p}_internal_node")
        rows.append((f"q{p}_ri", K.T_R, float(str(K.OPMODEL_RI)), pos, neg, -1, -1, -1))
        rows.append((f"q{p}_ro", K.T_R, float(str(K.OPMODEL_RO)), inner, out, -1, -1, -1))
        rows.append((f"q{p}_vcvs", K.T_VCVS, float(str(K.OPMODEL_GAIN)), inner, gid, pos, neg, -1))
        rows.append((f"q{p}_rf", K.T_R, rf, neg, out, -1, -1, -1))
    col = lambda k, dt: np.array([r[k] for r in rows], dtype=dt).reshape(-1)   # noqa: E731
    loads = 10 ** rng.uniform(2, 4, sites)
    load_a, load_b = (np.full(sites, gid), sid) if ideal_pads else (sid, np.full(sites, gid))
    a_id = np.concatenate([ra, load_a, col(3, np.int64)])
    b_id = np.concatenate([rb, load_b, col(4, np.int64)])
    index, kcl = first_appearance_numbering(a_id, b_id, gid)
    index = np.append(index, -1).astype(np.int32)      # the id -1 of "no control node" maps to ground
    type_ = np.concatenate([np.full(m_r, K.T_R, np.uint8), np.full(sites, K.T_A if ideal_pads else K.T_R, np.uint8),
                            col(1, np.uint8)])
    value = np.concatenate([np.full(m_r, float(resistance)), float(vdd) / loads if ideal_pads else loads,
                            col(2, np.float64)])
    dep = np.isin(type_, (K.T_VCVS, K.T_VCCS, K.T_CCVS, K.T_CCCS))
    c_id = np.concatenate([np.full(m_r + sites, -1), col(5, np.int64)])
    d_id = np.concatenate([np.full(m_r + sites, -1), col(6, np.int64)])
    cc = np.where(dep, index[c_id], K.UNUSED).astype(np.int32)
    dd = np.where(dep, index[d_id], K.UNUSED).astype(np.int32)
    drv = np.concatenate([np.full(m_r + sites, -1), col(7, np.int64)]).astype(np.int32)
    anom = (type_ != K.T_R) & (type_ != K.T_A)
    branch = np.full(len(type_), -1, np.int32)
    be = int(anom.sum())
    branch[anom] = np.arange(be, dtype=np.int32)
    table = ComponentTable(type_, value, index[a_id], index[b_id], cc, dd, drv, branch, kcl=kcl, be=be)
    named = {name: gid + 1 + k for k, name in enumerate(extra_names)}

    def encode(name):
        if name == "g":
            return gid
        if name in named:
            return named[name]
        if not name.startswith("n"):
            return None
        try:
            px, py = (int(t) for t in name[1:].split("_"))
        except ValueError:
            return None
        return px * N + py if 0 <= px < N and 0 <= py < N else None

    def decode(nid):
        return "g" if nid == gid else extra_names[nid - gid - 1] if nid > gid else f"n{nid // N}_{nid % N}"

    tail = [r[0] for r in rows]

    def names(k):
        k = int(k)
        return f"r{k}" if k < m_r else f"l{k - m_r}" if k < m_r + sites else tail[k - m_r - sites]

    anom_names = [names(k) for k in np.flatnonzero(anom)]
    net = TableNetlist(table, _LazyNodeMap(index[:-1], encode, decode, kcl), "g", names=names,
                       anomnum={name: k for k, name in enumerate(anom_names)})
    net._currents = anom_names
    return net


# --------------------------------------------------------------------------- sparse random networks
def random_network(nodes, degree=8, seed=0, decades=2.0, locality=None):
    """Connected random resistive network (north star: "random-network netlists"): `nodes` nodes, a
    spanning chain (node i to a random earlier node, which keeps it connected) plus random extra
    resistors up to the average `degree`; resistances 10**U(0, decades) ohm.  Node "g" is node 0
    and "1" is the last node.  Rows are numbered by the reference's first-appearance rule
    (nodal/nodal.py:249-257,283-287) over the emitted component order, i.e. NOT geometrically:
    the CSR's column indices and the halo sets of a row partition are irregular.

    locality=None: the partner of every edge is uniform over all nodes (an expander-like graph:
    every row block touches every other, the worst case for x gathers and halos).
    locality=w: partners are drawn within +-w of the node id (a banded random graph, the shape a
    placed-and-routed netlist has)."""
    rng = np.random.default_rng(seed)
    nodes = int(nodes)
    chain_a = np.arange(1, nodes, dtype=np.int64)
    if locality is None:
        chain_b = (rng.random(nodes - 1) * chain_a).astype(np.int64)          # uniform in [0, i)
    else:
        chain_b = np.maximum(0, chain_a - 1 - (rng.random(nodes - 1) * np.minimum(chain_a, locality)).astype(np.int64))
    extra = max(0, (degree * nodes) // 2 - (nodes - 1))
    ea = rng.integers(0, nodes, size=extra, dtype=np.int64)
    if locality is None:
        eb = rng.integers(0, nodes, size=extra, dtype=np.int64)
    else:
        eb = np.clip(ea + rng.integers(-locality, locality + 1, size=extra, dtype=np.int64), 0, nodes - 1)
    keep = ea != eb
    # interleave the chain and the extra resistors so that first-appearance order is not simply
    # the node order: component k of the chain is followed by its share of the extras
    a_id = np.concatenate([chain_a, ea[keep]])
    b_id = np.concatenate([chain_b, eb[keep]])
    order = rng.permutation(len(a_id))
    a_id, b_id = a_id[order], b_id[order]
    gid, pid = 0, nodes - 1
    index, kcl = first_appearance_numbering(a_id, b_id, gid)
    m = len(a_id)
    value = 10.0 ** rng.uniform(0.0, decades, size=m)
    table = ComponentTable(np.full(m, K.T_R, np.uint8), value, index[a_id], index[b_id], kcl=kcl, be=0)

    def encode(name):
        if name == "1":
            return pid
        if name == "g":
            return gid
        if not name.startswith("n"):
            return None
        try:
            nid = int(name[1:])
        except ValueError:
            return None
        return nid if 0 < nid < nodes - 1 else None

    def decode(nid):
        return "1" if nid == pid else "g" if nid == gid else f"n{nid}"

    return TableNetlist(table, _LazyNodeMap(index, encode, decode, kcl), "g", names=lambda k: f"r{k}")


# --------------------------------------------------------------------------- config C3
def random_opamp_network_rows(M=3968, P=2048, S=2048, V=64, seed=0, extra_degree=8):
    """Config C3 (SURVEY.md 8(d)): random connected resistive network with OPMODEL
    op-amps, E sources and VCVS; returns csv-style rows.

    Every E source sits behind a series resistor (1 extra node), every op-amp stage owns
    its output, inverting and internal nodes, every VCVS drives its own node, so the
    unknown count is  nodes (M + S + 3P + V) + branches (S + P + V) = M + 2S + 4P + 2V;
    the defaults give 16 384."""
    rng = np.random.default_rng(seed)
    rows = []
    node = lambda k: f"n{k}"  # noqa: E731
    k = 0
    for i in range(M):                      # spanning chain through ground keeps it connected
        other = "g" if i == 0 else node(int(rng.integers(0, i)))
        rows.append([f"r{k}", "R", repr(float(10 ** rng.uniform(0, 4))), node(i), other]); k += 1
    extra = max(0, (extra_degree * M) // 2 - M)
    ea = rng.integers(0, M, size=extra)
    eb = rng.integers(0, M, size=extra)
    ev = 10 ** rng.uniform(0, 4, size=extra)
    for x, y, v in zip(ea, eb, ev):
        if x != y:
            rows.append([f"r{k}", "R", repr(float(v)), node(int(x)), node(int(y))]); k += 1
    src_nodes = rng.choice(M, size=S + V, replace=False)
    for s in range(S):                      # stiff sources through a series resistor
        mid = f"s{s}"
        rows.append([f"rs{s}", "R", repr(float(10 ** rng.uniform(0, 2))), mid, node(int(src_nodes[s]))])
        rows.append([f"e{s}", "E", repr(float(rng.uniform(-10, 10))), mid, "g"])
    for p in range(P):                      # non-inverting stages: gain = 1 + rf/rg <= 100
        pos = node(int(rng.integers(0, M)))
        out, neg = f"o{p}", f"m{p}"
        rf = float(10 ** rng.uniform(2, 4))
        rg = rf / float(rng.uniform(0.5, 99.0))
        rows.append([f"q{p}", "OPMODEL", repr(rf), out, "g", pos, neg])
        rows.append([f"rg{p}", "R", repr(rg), neg, "g"])
        rows.append([f"rl{p}", "R", repr(float(10 ** rng.uniform(2, 4))), out, "g"])
    for v in range(V):
        tgt = f"v{v}"
        c1, c2 = node(int(rng.integers(0, M))), node(int(rng.integers(0, M)))
        rows.append([f"d{v}", "VCVS", repr(float(rng.uniform(-2, 2))), tgt, "g", c1, c2])
        rows.append([f"rv{v}", "R", repr(float(10 ** rng.uniform(1, 3))), tgt,
                     node(int(src_nodes[S + v]))])
    return rows


# --------------------------------------------------------------------------- config C4
def opamp_sweep_values(batch, seed=0):
    """Config C4: per-copy values of the 6 components of doc/opmodel_amplifier.csv in the
    stamping order v1, r1, q1_ri, q1_ro, q1_vcvs, q1_rf (SURVEY.md 8(d))."""
    rng = np.random.default_rng(seed)
    vals = np.empty((batch, 6))
    vals[:, 0] = rng.uniform(-5, 5, batch)            # v1   (E)
    vals[:, 1] = 10 ** rng.uniform(2, 5, batch)       # r1
    vals[:, 2] = 1e7 * rng.uniform(0.5, 2, batch)     # ri
    vals[:, 3] = 10 * rng.uniform(0.5, 2, batch)      # ro
    vals[:, 4] = 1e5 * rng.uniform(0.5, 2, batch)     # gain
    vals[:, 5] = 10 ** rng.uniform(2, 5, batch)       # rf
    return vals


OPAMP_AMPLIFIER_ROWS = [["q1", "OPMODEL", "1", "2", "g", "3", "1"],
                        ["v1", "E", "1", "3", "g"],
                        ["r1", "R", "1", "g", "1"]]
