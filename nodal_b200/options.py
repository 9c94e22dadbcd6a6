"""The keyword options of a Circuit parsed once (SolveOptions: its field defaults are the only place the
defaults are written; unknown keys are ignored) and the ordered candidates of its single-GPU sparse solve."""
from __future__ import annotations

import dataclasses
from typing import NamedTuple

import numpy as np

from . import constants as K
from . import schur
from . import source_schur
from . import sources


@dataclasses.dataclass(frozen=True)
class SolveOptions:
    """The options of Circuit(netlist, sparse, **options) that its solve paths read."""
    device: int | None = None
    distributed: bool = False
    csr_order: str = "sorted"
    atomic_stamp: bool = False
    check_connected: bool = False
    precond: str = "auto"
    rtol: float | None = None          # None: not given (spd_rtol / gmres_rtol)
    maxit: int | None = None
    amg: dict | None = None
    pcg_flags: int = 0
    auto_probe_iterations: int = 24
    auto_probe_min_rows: int = 50_000
    amg_graph_min_rows: int = 100_000
    multi_rhs: bool = True
    restart: int = 60
    gmres_fallback: bool = True
    dense_fallback_max_rows: int = 32768
    x0: np.ndarray | None = None
    eliminate_sources: bool | str = "auto"
    schur: bool = False
    schur_rtol: float | None = None    # None: rtol
    schur_refine: int = 5
    schur_max_branches: int = 8192

    # derived: SPD solver on one GPU; tolerances of all but GMRES, of GMRES, of the Schur paths' L solves
    spd_solver = property(lambda self: "pcg" if self.precond == "jacobi" else "amg")
    spd_rtol = property(lambda self: 1e-10 if self.rtol is None else self.rtol)
    gmres_rtol = property(lambda self: 1e-12 if self.rtol is None else self.rtol)
    inner_rtol = property(lambda self: self.spd_rtol if self.schur_rtol is None else self.schur_rtol)
    gmres_maxit = property(lambda self: self.maxit or 20000)
    amg_params = property(lambda self: self.amg or {})


_FIELDS = {f.name for f in dataclasses.fields(SolveOptions)}


def parse(options, sparse, table):
    """SolveOptions of Circuit(netlist, sparse, **options) on `table`.  Raises ValueError (or
    NotImplementedError for schur=True with distributed=True) on an invalid option.  precond,
    eliminate_sources and x0 are only checked for the sparse path, the only one that reads them."""
    kw = {k: v for k, v in options.items() if k in _FIELDS}
    for k in ("schur_refine", "schur_max_branches", "dense_fallback_max_rows", "auto_probe_iterations"):
        if k in kw:
            kw[k] = int(kw[k])
    opts = SolveOptions(**kw)
    if opts.schur is not True and opts.schur is not False:
        raise ValueError(f"schur must be True or False, got {opts.schur!r}")
    if opts.schur and not sparse:
        raise ValueError("schur=True needs sparse=True (the dense path already solves by LU)")
    if opts.schur and opts.distributed:
        raise NotImplementedError("the Schur-complement solve runs on one GPU (distributed=True is not supported)")
    if opts.schur_refine < 0:
        raise ValueError("schur_refine must be >= 0")
    if opts.schur_max_branches < 1:
        raise ValueError("schur_max_branches must be >= 1")
    if not sparse:
        return opts
    mode = opts.eliminate_sources
    if not (mode is True or mode is False or mode == "auto"):
        raise ValueError(f"eliminate_sources must be 'auto', True or False, got {mode!r}")
    if mode is True and not opts.distributed and table.facts()["present"] & ~sources._RAE and not opts.schur:
        raise ValueError("eliminate_sources=True needs a netlist of R, A and E rows only "
                         "(dependent sources cannot be eliminated; with schur=True they go through the "
                         "Schur complement of the reduced system)")
    if opts.precond not in ("auto", "jacobi", "amg"):
        raise ValueError(f"precond must be 'auto', 'jacobi' or 'amg', got {opts.precond!r}")
    if opts.x0 is not None and not opts.distributed:
        x0 = np.ascontiguousarray(opts.x0, dtype=np.float64)
        if x0.shape != (table.n,):
            raise ValueError(f"x0 must have {table.n} entries")
        opts = dataclasses.replace(opts, x0=x0)
    return opts


class Candidate(NamedTuple):
    """An exact sparse path: reason "" when the host lets it run, else why not (and Circuit.solve reports
    `declined` under info[key])."""
    path: str
    key: str
    reason: str
    declined: dict


def plan(table, opts):
    """The paths asked for, in the order Circuit.solve tries them: sources (R / A / E tables),
    source_schur (E and dependent rows, schur=True and eliminate_sources=True), schur (schur=True)."""
    out = []
    reason = sources.skip_reason(table, opts.eliminate_sources, opts.dense_fallback_max_rows)
    if reason is not None:
        out.append(Candidate("sources", "reduction", reason, dict(eliminated=False, reason=reason)))
    if (opts.schur and opts.eliminate_sources is True and table.has_type(K.T_E)
            and table.facts()["present"] & source_schur._DEP):
        reason = source_schur.skip_reason(table)
        out.append(Candidate("source_schur", "reduction", reason, dict(eliminated=False, applied=False, reason=reason)))
    if opts.schur:
        reason = schur.skip_reason(table, opts.schur_max_branches)
        out.append(Candidate("schur", "schur", reason,
                             dict(applied=False, branches=table.be, node_rows=table.kcl, reason=reason)))
    return out
