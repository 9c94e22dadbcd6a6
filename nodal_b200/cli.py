"""Shared pieces of the two console entry points (`nodal-solver`, `nodal-resistance`)."""
import argparse
import os
import sys

import nodal_b200 as n


def make_parser(description, file_help):
    """FILE plus -s/--sparse: the whole command line of both tools (reference
    nodal/solver.py:7-13, nodal/equiv.py:11-19)."""
    parser = argparse.ArgumentParser(description=description)
    parser.add_argument("netlist_path", metavar="FILE", help=file_help)
    parser.add_argument("-s", "--sparse", action="store_true", help="use a sparse matrix")
    # additions to the reference command line (both default to its behaviour)
    parser.add_argument("--precond", choices=("auto", "jacobi", "amg"), default="auto",
                        help="preconditioner of the sparse solve for resistor networks (auto: aggregation "
                             "AMG, Jacobi if that fails)")
    parser.add_argument("--check-connected", action="store_true",
                        help="with -s: fail on floating sub-circuits instead of printing what the "
                             "iterative solver returned")
    parser.add_argument("--eliminate-sources", choices=("auto", "on", "off"), default="auto",
                        help="with -s: solve R / A / E netlists by eliminating the voltage sources and running "
                             "the AMG-PCG on the reduced system (auto: above the dense-LU fallback size); "
                             "'on' with --schur: eliminate the voltage sources of a netlist with op-amps and "
                             "dependent sources, then solve the rest through the Schur complement")
    parser.add_argument("--schur", action="store_true",
                        help="with -s: solve netlists with op-amps and dependent sources through the Schur "
                             "complement of the branch rows (AMG on the resistor block, dense LU on the rest); "
                             "with --eliminate-sources on, of the rows left after the voltage sources are "
                             "eliminated")
    return parser


def circuit_options(options):
    """Keyword arguments for Circuit from the parsed command line."""
    kw = {}
    if options.sparse and options.precond != "auto":
        kw["precond"] = options.precond
    if options.sparse and options.check_connected:
        kw["check_connected"] = True
    mode = getattr(options, "eliminate_sources", "auto")
    if options.sparse and mode != "auto":
        kw["eliminate_sources"] = mode == "on"
    if options.sparse and getattr(options, "schur", False):
        kw["schur"] = True
    return kw


# Files at least this large go through the vectorised ingest (nodal_b200.ingest): same numbering,
# ~7 us per row less.  Smaller ones keep the reference's row-by-row objects.
FAST_INGEST_BYTES = 1 << 20


def load_netlist_or_exit(path):
    """Exit status 1 when the file does not exist (the error itself is logged by Netlist)."""
    try:
        if os.path.isfile(path) and str(path).endswith(".npz"):      # binary form, see ingest.save_table_netlist
            from nodal_b200.ingest import load_table_netlist
            return load_table_netlist(path)
        if os.path.isfile(path) and os.path.getsize(path) >= FAST_INGEST_BYTES:
            from nodal_b200.ingest import read_table_netlist
            try:
                return read_table_netlist(path)
            except Exception:       # malformed input: let the row-by-row parser report it its way
                pass
        return n.Netlist(path)
    except FileNotFoundError:
        sys.exit(1)
