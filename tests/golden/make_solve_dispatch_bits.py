#!/usr/bin/env python
"""Record what Circuit.solve computes on every sparse solve path, for tests/test_gpu_solve_dispatch_bits.py.

Usage (on a GPU, with the tree whose results are the reference):
    python tests/golden/make_solve_dispatch_bits.py [out.json]

Writes tests/golden/solve_dispatch_bits.json (or `out.json`): for every case of CASES, the SHA-256 of
the float64 bytes of Solution.result (a few leading values for diagnosis) and Solution.stats with every
key ending in "_ms" removed at every depth, dumped as JSON with sorted keys.  The cases cover the
choice of path (AMG / Jacobi / probe, source elimination, Schur complement, both, the GMRES and dense-LU
fall-backs) and what each declined path reports, so a change to how the path is chosen that keeps its
behaviour must leave all of them unchanged.
"""
import copy
import hashlib
import json
import os
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

PORTS = [("1", "g"), ("n10_10", "g"), ("n3_150", "n120_7"), ("n199_199", "n0_0"), ("1", "1")]


def digest(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(), "n": int(a.size), "head": [float(v) for v in a[:4]]}


def _plain(v):
    """The stats without timings: keys ending in "_ms" dropped at every depth, numpy scalars as Python."""
    if isinstance(v, dict):
        return {str(k): _plain(x) for k, x in v.items() if not str(k).endswith("_ms")}
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    if isinstance(v, np.generic):
        return v.item()
    return v


def stats_text(stats):
    return json.dumps(_plain(stats), sort_keys=True)


def _probed_grid():
    from nodal_b200 import generators as gen
    net = copy.deepcopy(gen.grid2d(200))
    net.process_component(["a1", "A", "1", "1", "g"])
    return net


def _doc_netlist(name):
    import nodal_b200 as n
    from helpers import golden, write_csv
    rows = golden("doc_netlists.json")[name]["rows"]
    path = os.path.join(tempfile.mkdtemp(), "netlist.csv")
    return n.Netlist(write_csv(rows, path))


def _source_loop():
    import nodal_b200 as n
    from helpers import write_csv
    from oracle import mna_oracle as orc
    rows = orc.grid2d_rows(40) + [["v1", "E", "1", "n0_0", "g"], ["v2", "E", "1", "n0_0", "g"],
                                  ["a1", "A", "1e-3", "g", "n20_20"]]
    return n.Netlist(write_csv(rows, os.path.join(tempfile.mkdtemp(), "loop.csv")))


def _small_rae():
    from nodal_b200 import generators as gen
    return gen.power_grid(40, 8, vdd=1.0, load=1e-3, seed=1)


def _power_grid():
    from nodal_b200 import generators as gen
    return gen.power_grid(300, 20, vdd=1.0, load=1e-4, seed=0)


def _amplifier(ideal_pads=False):
    from nodal_b200 import generators as gen
    return gen.amplifier_grid(64, 8, seed=0, ideal_pads=ideal_pads)


def _x0(n):
    return np.random.default_rng(11).uniform(0.0, 1e-2, n)


# name -> (netlist factory, Circuit options); "x0" is filled in with _x0 of the table's size
CASES = {
    "grid200_auto": (_probed_grid, {}),
    "grid200_jacobi": (_probed_grid, dict(precond="jacobi")),
    "grid200_amg": (_probed_grid, dict(precond="amg")),
    "grid200_x0": (_probed_grid, dict(x0=True)),
    "grid200_x0_jacobi": (_probed_grid, dict(x0=True, precond="jacobi")),
    "grid200_first_touch": (_probed_grid, dict(csr_order="first_touch")),
    "grid200_schur_no_branches": (_probed_grid, dict(schur=True)),
    "power_grid300_auto": (_power_grid, {}),
    "power_grid300_x0": (_power_grid, dict(x0=True)),
    "power_grid300_no_elimination": (_power_grid, dict(eliminate_sources=False)),
    "power_grid40_below_limit": (_small_rae, {}),
    "source_loop_eliminate": (_source_loop, dict(eliminate_sources=True)),
    "amplifier64_schur": (_amplifier, dict(schur=True)),
    "amplifier64_schur_refine0": (_amplifier, dict(schur=True, schur_refine=0)),
    "amplifier64_ideal_source_schur": (lambda: _amplifier(True), dict(schur=True, eliminate_sources=True)),
    "amplifier64_ideal_source_schur_refine0": (lambda: _amplifier(True),
                                               dict(schur=True, eliminate_sources=True, schur_refine=0)),
    "amplifier64_ideal_schur_auto": (lambda: _amplifier(True), dict(schur=True)),
    "test_1_source_schur": (lambda: _doc_netlist("test_1.csv"), dict(schur=True, eliminate_sources=True)),
    "test_1_sparse": (lambda: _doc_netlist("test_1.csv"), {}),
}


def run_case(name):
    """(digest of Solution.result, stats text) of one case."""
    import nodal_b200 as n
    make, opts = CASES[name]
    net = make()
    opts = dict(opts)
    if opts.get("x0"):
        opts["x0"] = _x0(net.table().n)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        sol = n.Circuit(net, sparse=True, **opts).solve()
    return digest(sol.result), stats_text(sol.stats)


def ports(pairs):
    """(digest of the resistances, stats text) of equivalent_resistances over `pairs` on grid2d(200): several
    pairs share one hierarchy, a single one goes through the solve of one right-hand side."""
    from nodal_b200 import equiv
    from nodal_b200 import generators as gen
    values = equiv.equivalent_resistances(gen.grid2d(200), pairs, sparse=True)
    return digest(values), stats_text(equiv.equivalent_resistances.last_stats)


def main():
    out = {}
    for name in CASES:
        d, s = run_case(name)
        out[name] = {"result": d, "stats": s}
        print(name, d["sha256"][:16], s[:160], flush=True)
    for name, pairs in (("equivalent_resistances", PORTS), ("equivalent_resistances_single", PORTS[1:2])):
        d, s = ports(pairs)
        out[name] = {"result": d, "stats": s}
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "solve_dispatch_bits.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    main()
