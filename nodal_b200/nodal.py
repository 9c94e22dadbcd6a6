"""Host-side mirror of the reference's central module (nodal/nodal.py) for the MNA hot path.

Same classes and call signatures as the reference --

    from nodal_b200 import Circuit, Netlist
    solution = Circuit(Netlist("netlist.csv"), sparse=True).solve()
    print(solution)

-- but numbering produces a struct-of-arrays component table, stamping and the
linear solve run as sm_100a CUDA kernels through libnodal_b200.so, and nothing on
this path falls back to numpy / scipy arithmetic.

Reference lines mirrored: find_ground_node nodal.py:30-42, build_opmodel :45-85,
is_connected :88-105, Component :112-178, Netlist :181-296, Circuit :299-398,
Solution :401-434.
"""
from __future__ import annotations

import csv
import logging
import warnings

import numpy as np

from . import constants as c
from . import models
from . import dist as ndist
from . import dist_sources
from . import options as solve_options
from . import schur
from . import source_schur
from . import sources
from .table import ComponentTable

logging.basicConfig(level=logging.ERROR)  # as the reference does at import (nodal.py:27)

__all__ = ["find_ground_node", "build_opmodel", "is_connected", "UnconnectedCircuitError",
           "Component", "Netlist", "Circuit", "Solution", "c", "models", "np", "logging"]


def find_ground_node(degrees):
    """Node used as the 0 V reference: "g" when present, otherwise the first node
    (insertion order) with the largest number of attached leads."""
    if "g" in degrees:
        ground = "g"
    else:
        ground = max(degrees.keys(), key=degrees.__getitem__)
    logging.debug(f"ground node-> {ground}")
    return ground


def build_opmodel(data):
    """Expand an OPMODEL row [name, "OPMODEL", rf, out, gnd, pos, neg] into the
    macro model: input resistor, output resistor, VCVS and (unless rf is the
    string "0") the feedback resistor.  Values go through str() exactly as in the
    reference so that float() later parses the same digits."""
    name, rf = data[c.NCOL], data[c.VCOL]
    out, gnd, pos, neg = data[c.ACOL], data[c.BCOL], data[c.CCOL], data[c.DCOL]
    inner = f"{name}_internal_node"
    parts = [
        [f"{name}_ri", "R", str(c.OPMODEL_RI), pos, neg],
        [f"{name}_ro", "R", str(c.OPMODEL_RO), inner, out],
        [f"{name}_vcvs", "VCVS", str(c.OPMODEL_GAIN), inner, gnd, pos, neg],
    ]
    if rf != "0":
        parts.append([f"{name}_rf", "R", rf, neg, out])
    else:
        assert neg == out
    return parts


def is_connected(netlist):
    """True when every node can be reached from ground through component leads
    (control nodes do not count).  Diagnostic for singular systems only."""
    adjacency = {node: set() for node in netlist.degrees}
    for comp in netlist.components.values():
        adjacency[comp.anode].add(comp.bnode)
        adjacency[comp.bnode].add(comp.anode)
    seen = {netlist.ground}
    frontier = [netlist.ground]
    while frontier:
        nxt = []
        for node in frontier:
            for other in adjacency[node]:
                if other not in seen:
                    seen.add(other)
                    nxt.append(other)
        frontier = nxt
    return len(seen) == len(adjacency)


class UnconnectedCircuitError(Exception):
    pass


class Component:
    """One electrical component, built from a csv row (list of str).

    Attributes: name, type, value, anode, bnode, pos_control, neg_control and,
    for dependent sources only, driver (None unless current controlled).
    Raises ValueError on malformed rows.
    """

    def __init__(self, data):
        self.check_input(data)
        self.name = data[c.NCOL]
        self.type = data[c.TCOL]
        self.value = float(data[c.VCOL])
        self.anode = data[c.ACOL]
        self.bnode = data[c.BCOL]
        self.pos_control = None
        self.neg_control = None
        if self.type in c.NODE_TYPES_DEP:
            self.pos_control = data[c.CCOL]
            self.neg_control = data[c.DCOL]
            self.driver = data[c.PCOL] if self.type in c.NODE_TYPES_CC else None

    def check_input(self, data):
        n_fields = len(data)
        if n_fields == 0 or data[0][0] == "#":
            return
        key = data[c.NCOL]
        assert type(key) == str
        if n_fields < 5:
            raise ValueError(f"Missing arguments for component {key}")
        ctype = data[c.TCOL]
        if ctype not in c.NODE_TYPES:
            raise ValueError(f"Unknown type {ctype} for component {key}")
        expected = c.NODE_ARGS_NUMBER[ctype]
        if n_fields != expected:
            raise ValueError(
                f"Wrong number of arguments for component {key}: expected {expected}, got {n_fields}")
        try:
            float(data[c.VCOL])
        except ValueError:
            raise ValueError("Bad input: expected a number for component value "
                             f"of {key}, got {data[c.VCOL]} instead")


class Netlist:
    """Reads a netlist from a .csv file and numbers its unknowns.

    Attributes (same meaning as the reference): nums, degrees, anomnum,
    components, component_keys, ground, nodenum, opmodel_equivalents.
    ``table()`` additionally returns the struct-of-arrays component table the
    stamp kernel consumes.
    Raises FileNotFoundError / ValueError like the reference.
    """

    def __init__(self, path):
        self.nums = {"components": 0, "anomalies": 0, "be": 0, "kcl": 0, "opamps": 0}
        self.degrees = {}
        self.anomnum = {}
        self.components = {}
        self.component_keys = []
        self.ground = None
        self.nodenum = {}
        self.opmodel_equivalents = []
        self.read_netlist(path)

    # ---- numbering -------------------------------------------------------------
    def process_component(self, data):
        """Register one csv row: component record, node degrees, branch number."""
        if data == [] or data[0][0] == "#":
            return
        if data[c.TCOL] == "OPMODEL":           # expanded now, registered after all rows
            self.opmodel_equivalents.extend(build_opmodel(data))
            return
        comp = Component(data)
        key = data[c.NCOL]
        self.component_keys.append(key)         # duplicates are kept on purpose (stamping order)
        self.components[key] = comp
        self.nums["components"] += 1
        leads = [data[c.ACOL], data[c.BCOL]]
        unseen = [node for node in leads if node not in self.degrees]
        if data[c.TCOL] in c.NODE_TYPES_ANOM:
            self.anomnum[key] = self.nums["anomalies"]
            self.nums["anomalies"] += 1
        for node in unseen:
            self.degrees[node] = 0
        for node in leads:
            self.degrees[node] += 1

    def read_netlist(self, path):
        try:
            handle = open(path, "r")
        except FileNotFoundError:
            logging.error(f"File '{path}' not found.")
            raise
        with handle:
            for row in csv.reader(handle, skipinitialspace=True):
                self.process_component(row)
        for row in self.opmodel_equivalents:
            self.process_component(row)
        self._number_nodes()

    def _number_nodes(self):
        self.ground = find_ground_node(self.degrees)
        self.nodenum = {}
        for node in self.degrees:
            if node != self.ground:
                self.nodenum[node] = len(self.nodenum)
        assert len(self.nodenum) == len(self.degrees) - 1
        logging.debug(f"nodenum={self.nodenum}")
        self.nums["kcl"] = len(self.nodenum)
        self.nums["be"] = self.nums["anomalies"]
        logging.debug(f"nums={self.nums}")
        logging.debug(f"anomnum={self.anomnum}")

    # ---- B200 build: component table --------------------------------------------
    def is_resistive(self):
        return all(comp.type == "R" for comp in self.components.values())

    def table(self) -> ComponentTable:
        """Component table in stamping order.  Goes through the same dispatch as the
        reference's build_model (nodal.py:357-390) with a recorder in place of G."""
        return self.table_and_currents()[0]

    def table_and_currents(self):
        rec = models.StampRecorder(self)
        self._dispatch(rec)
        return rec.finish(), rec.currents

    def _dispatch(self, G):
        nums, anomnum, nodenum = self.nums, self.anomnum, self.nodenum
        ground, components = self.ground, self.components
        A, currents = G.rhs_proxy, G.currents
        for key in self.component_keys:
            comp = components[key]
            i = nodenum[comp.anode] if comp.anode != ground else None
            j = nodenum[comp.bnode] if comp.bnode != ground else None
            args = (comp, i, j, ground, G, A, currents, anomnum, nums, nodenum)
            kind = comp.type
            if kind == "R":
                models.write_R(comp, i, j, ground, G)
            elif kind == "A":
                models.write_A(comp, i, j, ground, A)
            elif kind == "E":
                models.write_E(*args)
            elif kind == "VCCS":                 # the reference stamps VCCS as a VCVS (nodal.py:377-378)
                models.write_VCVS(*args)
            elif kind == "VCVS":
                models.write_VCVS(*args)
            elif kind == "CCVS":
                models.write_CCVS(*args, components)
            elif kind == "CCCS":
                models.write_CCCS(*args, components)
            elif kind == "OPAMP":
                raise NotImplementedError
            else:
                raise ValueError(f"Unknown component type: {kind}")


class Circuit:
    """Builds and solves the MNA system  G e = A  of a Netlist on the GPU.

    ``sparse=False``: dense G, blocked FP64 LU with partial pivoting (replaces
    numpy.linalg.solve).  ``sparse=True``: CSR G (replaces scipy spsolve); on one
    GPU the exact paths asked for run in this order, the first that qualifies
    solves (options.plan, see solve() for what the others report): the
    elimination of the voltage sources (sources.py), with ``schur=True,
    eliminate_sources=True`` the elimination then the Schur complement
    (source_schur.py), with ``schur=True`` the Schur complement of the branch
    rows (schur.py); then PCG for R/A netlists, restarted GMRES otherwise.
    ``distributed=True``: dist_sources.py for R/A/E netlists, else dist.GridRunner.
    The options are parsed once (``circuit.opts``); ``circuit.options`` is the
    dict the caller passed.

    Attributes as in the reference: netlist, sparse, G, A, currents.  G and A
    live in HBM; ``G`` is a torch tensor (dense) or a DeviceCSR, and
    ``np.asarray(circuit.G)`` / ``circuit.G.tocsr()`` / ``circuit.A_host`` give host
    copies.
    """

    def __init__(self, netlist, sparse=False, **options):
        if not isinstance(netlist, Netlist):
            raise TypeError("Input isn't a netlist")
        self.netlist = netlist
        self.sparse = sparse
        self.options = options
        self.stats = {}
        self.G, self.A, self.currents = self.build_model()

    # ---- assembly ---------------------------------------------------------------
    def build_model(self):
        from .device import Device
        table, currents = self.netlist.table_and_currents()
        self.opts = opts = solve_options.parse(self.options, self.sparse, table)
        table.validate()
        self.table = table
        dev = Device.get(opts.device)
        self._dev = dev
        self._dist = None
        self._dsrc = None
        self._dtab = None
        self._G_sorted = None
        self._plan = []
        if opts.distributed:
            G, A = self._build_distributed(dev, table)
        elif self.sparse:
            self._plan = solve_options.plan(table, opts)
            # the paths left after the host checks read the table's device columns (sources.py, schur.py,
            # source_schur.py)
            if any(not step.reason for step in self._plan):
                self._dtab = dev.upload_table(table)
            # csr_order="first_touch": G's columns in the order the reference's G.tocsr() has before its
            # solve (nodal.py:396-397); the solve then works on the sorted form, as spsolve sorts in place
            G, A = dev.assemble_csr(table, dtab=self._dtab, order=opts.csr_order)
            if opts.csr_order != "sorted":
                self._G_sorted = dev.assemble_csr(table)[0]
        else:
            G, A = dev.assemble_dense(table, atomic=bool(opts.atomic_stamp))
        logging.debug(f"currents={currents}")
        return [G, A, currents]

    def _build_distributed(self, dev, table):
        """Row-partitioned form (one process per GPU under torchrun, torch.distributed initialised
        with the nccl backend): every rank holds the netlist, uploads the table, selects the
        components touching its rows on the device and builds its rows of G only.  G is then a
        LocalRows view (the rank's rows, global columns), A the rank's slice of the right-hand side."""
        import torch.distributed as tdist
        if not self.sparse:
            raise ValueError("distributed=True needs sparse=True (the dense LU is single-GPU)")
        if not (tdist.is_available() and tdist.is_initialized()):
            raise RuntimeError("distributed=True needs an initialised torch.distributed process group")
        rank, world = tdist.get_rank(), tdist.get_world_size()
        if sources.skip_reason(table, True, 0) is not None:
            # R / A / E netlists with E rows: through the row-partitioned elimination of the sources (dist_sources.py)
            self._dsrc = dist_sources.DistSources(self, dev, table, rank, world)
            return self._dsrc.G, self._dsrc.A
        runner = ndist.GridRunner(dev, table, 0, rank, world, rtol=self.opts.spd_rtol,
                                  precond="jacobi" if self.opts.precond == "jacobi" else "amg",
                                  amg=self.opts.amg, solver=ndist.shared_solver(dev, rank, world))
        indptr, indices, data, rhs = runner.assemble_from_host()
        self._dist = runner
        return ndist.LocalRows(table.n, runner.bounds, rank, indptr, indices, data), rhs

    @property
    def A_host(self):
        return self.A.cpu().numpy()

    @property
    def G_host(self):
        if self.sparse:
            return self.G.tocsr()
        return self.G.cpu().numpy()

    # ---- solve ------------------------------------------------------------------
    def _sorted_G(self):
        """G, sorted (csr_order="first_touch" sorts before a solve reads G, as spsolve does: SURVEY.md app. C-5)."""
        if self._G_sorted is not None:
            self.G, self._G_sorted = self._G_sorted, None
        return self.G

    def _device_solve(self, rhs, amg=None):
        """x, info for G x = rhs on the device (rhs is a device tensor; dense G is not modified).
        Distributed circuits: rhs and x are the rank's slices."""
        dev, opts = self._dev, self.opts
        if not self.sparse:
            return dev.lu_solve(self.G.clone(), rhs)
        if self._dsrc is not None:
            raise NotImplementedError("the row-partitioned solve of a netlist with voltage sources is implemented "
                                      "for solve() only")
        # R / A netlists: precond "auto" = AMG-PCG with a Jacobi-PCG retry if the hierarchy cannot be built or
        # the solve does not converge (singular systems behave as on the Jacobi path); "amg" / "jacobi" force one
        kind = opts.spd_solver if self.table.is_spd_structured() else "gmres"
        G = self._sorted_G()
        if self._dist is not None:
            if kind == "gmres":
                raise NotImplementedError("row-partitioned solve is implemented for R / A netlists")
            return ndist.amg_then_jacobi(self._dist.pcg, G, rhs, opts)
        if kind in ("amg", "pcg"):
            warm = None if opts.x0 is None else dev.to_device(opts.x0)      # Circuit(..., x0=): SURVEY.md section 5
            return self._spd_solve(G, rhs, kind, opts.spd_rtol, warm, amg)
        x, info = dev.gmres(G, rhs, rtol=opts.gmres_rtol, restart=opts.restart, maxit=opts.gmres_maxit)
        # The reference's sparse path is a direct solve, exact for any non-singular MNA system; the
        # diagonally preconditioned GMRES can stall on indefinite systems with many source /
        # op-amp rows.  Rather than handing back an unconverged iterate, systems that fit the dense
        # LU go through it; larger ones are reported (NaNs + warning in solve(), as for breakdown).
        if info["status"] == 2 and opts.gmres_fallback:
            limit = opts.dense_fallback_max_rows
            if G.n <= limit:
                x, lu = dev.lu_solve(dev.csr_to_dense(G), rhs)
                lu.update(solver="lu (after gmres did not converge)", gmres_iterations=info["iterations"],
                          gmres_relres=info["relres"], relres=None)
                if lu["status"] == 1:
                    lu["status"] = 3            # singular: reported like a breakdown (NaNs + warning)
                return x, lu
            info["status"] = 3
            info["note"] = (f"gmres did not converge (relres {info['relres']:.2e}) and the system has more than "
                            f"{limit} rows (dense fallback limit)")
        return x, info

    def _spd_solve(self, G, rhs, kind, rtol, warm, amg=None):
        """x, info for an SPD DeviceCSR G (R / A netlists, or the reduced system of csrc/sources.cu) on
        one GPU: "amg" (with the "auto" Jacobi probe and the Jacobi-PCG retry) or "pcg"."""
        dev, opts = self._dev, self.opts
        if kind == "amg" and amg is None and warm is None and opts.precond == "auto":
            # "auto": which preconditioner pays depends on the graph, not on its size -- on a 4 M-node
            # expander-like random network Jacobi-PCG needs 98 iterations (43 ms) and the AMG hierarchy
            # 265 ms; on a banded random network of the same size it is 4 616 iterations (1.9 s)
            # against 68 (156 ms); grids are the second kind.  A short Jacobi-PCG probe tells them
            # apart: if 24 iterations gained two digits it will finish in ~100, otherwise its iterate
            # is the initial guess of the AMG solve.
            probe_its = opts.auto_probe_iterations
            if G.n >= opts.auto_probe_min_rows and probe_its > 0:
                x0, info0 = dev.pcg(G, rhs, rtol=rtol, maxit=probe_its, flags=opts.pcg_flags)
                if info0["status"] == 0:
                    info0["auto"] = "jacobi (converged inside the probe)"
                    return x0, info0
                if info0["status"] == 2 and info0["relres"] <= 1e-2:
                    x, info = dev.pcg(G, rhs, rtol=rtol, maxit=opts.maxit, x0=x0, flags=opts.pcg_flags)
                    info["iterations"] += info0["iterations"]
                    info["auto"] = f"jacobi (probe relres {info0['relres']:.1e})"
                    if info["status"] == 0:
                        return x, info
                    x0 = x
                elif info0["status"] != 2 or not np.isfinite(info0["relres"]):
                    x0 = None                                  # breakdown in the probe: start AMG from zero
                x, info = self._amg_solve(G, rhs, None, rtol, x0)
                if x0 is not None:
                    info["auto"] = f"amg (probe relres {info0['relres']:.1e})"
                    info["iterations_probe"] = info0["iterations"]
                return x, info
        if kind == "amg":
            return self._amg_solve(G, rhs, amg, rtol, warm)
        return dev.pcg(G, rhs, rtol=rtol, maxit=opts.maxit, flags=opts.pcg_flags, x0=warm)

    def _amg_solve(self, G, rhs, amg, rtol, x0):
        """AMG-preconditioned CG on one GPU; Jacobi-PCG retry unless precond="amg" was forced."""
        dev, opts = self._dev, self.opts
        from . import _lib
        try:
            if amg is not None:
                x, info = amg.solve(rhs, rtol=rtol, maxit=opts.maxit, x0=x0)
            elif G.n >= opts.amg_graph_min_rows:
                # large systems: the graph-captured form (csrc/dist_amg.cu with one rank):
                # one CUDA graph per iteration, no host round trip inside the iteration
                g = G
                bounds = np.array([0, g.n], dtype=np.int32)
                x, info = ndist.single_solver(dev).solve_amg(
                    g.n, bounds, g.indptr, g.indices, g.data, rhs, rtol=rtol, maxit=opts.maxit,
                    x0=x0, **opts.amg_params)
            else:
                x, info = dev.amg_pcg(G, rhs, rtol=rtol, maxit=opts.maxit, x0=x0, **opts.amg_params)
            if info["status"] == 0 or opts.precond == "amg":
                return x, info
            first = f"amg_pcg status {info['status']} after {info['iterations']} iterations"
        except _lib.NodalLibraryError as err:
            if opts.precond == "amg":
                raise
            first = str(err)
        x, info = dev.pcg(G, rhs, rtol=rtol, maxit=opts.maxit, flags=opts.pcg_flags)
        info["fallback_from_amg"] = first
        return x, info

    def is_connected(self):
        """Every node reaches ground through component leads (the reference's is_connected,
        nodal.py:88-105), decided on the device from the component table."""
        _, reached, _ = self._dev.connected_components(self.table)
        return reached == self.table.kcl + 1

    def solve(self):
        """Raises numpy.linalg.LinAlgError (singular dense system) or
        UnconnectedCircuitError (floating nodes), as the reference does.  The sparse path
        mirrors scipy (no exception; a Krylov solver even returns a finite solution when the
        singular system is consistent) unless the Circuit was built with check_connected=True:
        then the lead graph is checked on the device first and an unconnected circuit raises
        UnconnectedCircuitError like the dense path.

        On one GPU the sparse solve runs the candidates of options.plan in order (sources,
        source_schur, schur; a path's solve(circuit) gives (x, info), or (None, stats) when it
        declines) and _device_solve when none solves.  The stats of a declined sources or
        source_schur go under info["reduction"] (the two are exclusive by table content), those of
        a declined schur under info["schur"], never over a key the path which solved set (the schur
        stats of a successful source_schur stay); a path not asked for leaves no key."""
        if self.sparse and self.opts.check_connected and not self.is_connected():
            logging.error("Model error: unconnected circuit")
            raise UnconnectedCircuitError
        if self._dsrc is not None:
            x, info = self._dsrc.solve()            # dist_sources.py: x whole on every rank
        elif self.sparse and self._dist is None:
            self._sorted_G()
            declined = {}
            for step in self._plan:
                x, info = _PATHS[step.path].solve(self) if not step.reason else (None, dict(step.declined))
                if x is not None:
                    break
                declined[step.key] = info
            else:
                x, info = self._device_solve(self.A)
            for key, stats in declined.items():
                info.setdefault(key, stats)
        else:
            x, info = self._device_solve(self.A)
        if self.sparse:
            e = self._dist_gather(x) if self._dist is not None else x.cpu().numpy()
            if info["status"] != 0:
                # the reference's sparse path does not raise on singular systems: scipy warns
                # (MatrixRankWarning) and returns NaNs.  Mirror that.
                warnings.warn(f"sparse solve did not converge ({info})", RuntimeWarning)
                if info["status"] == 3 or not np.all(np.isfinite(e)):
                    e = np.full_like(e, np.nan)
        else:
            if info["status"] == 1:
                if not self.is_connected():
                    logging.error("Model error: unconnected circuit")
                    raise UnconnectedCircuitError
                logging.error("Model error: matrix is singular")
                raise np.linalg.LinAlgError("Singular matrix")
            e = x.cpu().numpy()
        self.stats = info
        sol = Solution(e, self.netlist, self.currents)
        sol.stats = info
        return sol

    def _dist_gather(self, x_local):
        """The whole solution vector on the host of every rank (slices all-gathered on the device)."""
        import torch.distributed as tdist
        torch, run = self._dev.torch, self._dist
        world = run.world
        sizes = np.diff(run.bounds).astype(np.int64)
        if world == 1:
            return x_local.cpu().numpy()
        pad = int(sizes.max())
        mine = torch.zeros(pad, dtype=torch.float64, device=self._dev.dev)
        mine[: x_local.numel()] = x_local
        full = torch.empty(world * pad, dtype=torch.float64, device=self._dev.dev)
        tdist.all_gather_into_tensor(full, mine)
        host = full.cpu().numpy().reshape(world, pad)
        return np.concatenate([host[k, : sizes[k]] for k in range(world)])

    def port_resistances(self, pairs):
        """e(a) - e(b) for a 1 A source from b to a, for every (a, b) in `pairs`, against the
        matrix assembled once (SURVEY.md section 8(f) rank 4: many-port equivalent resistance).
        Only the two potentials of a pair leave the device.  The AMG hierarchy is built once
        and shared by all right-hand sides."""
        dev, torch = self._dev, self._dev.torch
        n = self.table.n
        net = self.netlist
        run = self._dist
        lo, hi = (int(run.bounds[run.rank]), int(run.bounds[run.rank + 1])) if run is not None else (0, n)

        def row(node):
            return c.GROUND if node == net.ground else net.nodenum[node]

        def value_at(x, i):
            if i == c.GROUND:
                return 0.0
            if run is None or run.world == 1:
                return float(x[i - lo])
            import torch.distributed as tdist
            v = torch.zeros(1, dtype=torch.float64, device=dev.dev)
            if lo <= i < hi:
                v[0] = x[i - lo]
            tdist.broadcast(v, src=int(np.searchsorted(run.bounds, i, side="right") - 1))
            return float(v.item())

        amg = None
        pairs = list(pairs)
        # several right-hand sides share one hierarchy; a single solve goes through _device_solve's
        # own choice (auto probe, graph-captured form for large systems)
        if self.sparse and run is None and self.table.is_spd_structured() and self.opts.spd_solver == "amg" \
                and len(pairs) > 1:
            from . import _lib
            try:
                amg = dev.amg(self.G, **self.opts.amg_params)
            except _lib.NodalLibraryError:
                if self.opts.precond == "amg":
                    raise
                amg = None             # _device_solve retries per right-hand side and falls back to Jacobi
        values, stats = [], []
        try:
            if amg is not None and self.opts.multi_rhs:
                # several ports against one hierarchy: batches of up to 8 right-hand sides advance
                # together, every level operator is read once per sweep for the whole batch
                # (csrc/amg_multi.cu); a batch that does not converge is redone pair by pair below
                rows_of = [(row(a), row(b)) for a, b in pairs]
                todo = [k for k, (ia, ib) in enumerate(rows_of) if ia != ib]
                done = {}
                for start in range(0, len(todo), 8):
                    batch = todo[start:start + 8]
                    rhs = dev.zeros(max(2, len(batch) * n), torch.float64)[: len(batch) * n].view(len(batch), n)
                    for j, k in enumerate(batch):
                        ia, ib = rows_of[k]
                        if ia != c.GROUND:
                            rhs[j, ia] = 1.0
                        if ib != c.GROUND:
                            rhs[j, ib] = -1.0
                    xs, infos = amg.solve_multi(rhs, rtol=self.opts.spd_rtol, maxit=self.opts.maxit)
                    for j, k in enumerate(batch):
                        if infos[j]["status"] == 0:
                            ia, ib = rows_of[k]
                            ea = float(xs[j, ia]) if ia != c.GROUND else 0.0
                            eb = float(xs[j, ib]) if ib != c.GROUND else 0.0
                            done[k] = (ea - eb, infos[j])
                if len(done) == len(todo):
                    for k, (ia, ib) in enumerate(rows_of):
                        if ia == ib:
                            values.append(0.0)
                            stats.append(dict(solver="none", status=0, iterations=0))
                        else:
                            values.append(done[k][0])
                            stats.append(done[k][1])
                    self.stats = stats
                    return values
            for a, b in pairs:
                ia, ib = row(a), row(b)
                if ia == ib:
                    values.append(0.0)
                    stats.append(dict(solver="none", status=0, iterations=0))
                    continue
                rhs = dev.zeros(max(2, hi - lo), torch.float64)[: hi - lo]
                if ia != c.GROUND and lo <= ia < hi:
                    rhs[ia - lo] = 1.0
                if ib != c.GROUND and lo <= ib < hi:
                    rhs[ib - lo] = -1.0
                x, info = self._device_solve(rhs, amg=amg)
                if not self.sparse and info["status"] == 1:
                    raise np.linalg.LinAlgError("Singular matrix")
                if self.sparse and info["status"] != 0:
                    warnings.warn(f"sparse solve did not converge ({info})", RuntimeWarning)
                values.append(value_at(x, ia) - value_at(x, ib))
                stats.append(info)
        finally:
            if amg is not None:
                amg.close()
        self.stats = stats
        return values


_PATHS = {"sources": sources, "source_schur": source_schur, "schur": schur}


class Solution:
    """Result of a solve: ``result`` holds the kcl node potentials followed by the
    branch currents.  Printable, same layout as the reference."""

    def __init__(self, result, netlist, currents):
        self.result = result
        self.nodenum = netlist.nodenum
        self.nums = netlist.nums
        self.currents = currents
        self.ground = netlist.ground
        self.anomnum = netlist.anomnum
        self.stats = {}

    # ---- bulk access (SURVEY.md 8(f) rank 4): arrays instead of a line per node -----------
    def potentials(self):
        """Node potentials in row order (`nodenum[name]` indexes it); ground is 0 V."""
        return self.result[: self.nums["kcl"]]

    def branch_currents(self):
        """Currents of the anomalous branches in `anomnum` order."""
        return self.result[self.nums["kcl"]:]

    def save(self, path, names=False):
        """Binary export (numpy .npz): result, kcl, ground and, with names=True, the node and
        branch labels in row order.  Printing a 16 M-node solution sorts and formats every name."""
        payload = dict(result=np.asarray(self.result), kcl=np.int64(self.nums["kcl"]),
                       ground=np.array(str(self.ground)))
        if names:
            order = sorted(self.nodenum, key=self.nodenum.get)
            payload["nodes"] = np.array(order, dtype=str)
            payload["branches"] = np.array(sorted(self.anomnum, key=self.anomnum.get), dtype=str)
        np.savez(path, **payload)

    def __str__(self):
        lines = [f"Ground node: {self.ground}"]
        for name in sorted(self.nodenum):
            lines.append(f"e({name}) \t= {self.result[self.nodenum[name]]}")
        for name in sorted(self.anomnum):
            lines.append(f"i({name}) \t= {self.result[self.nums['kcl'] + self.anomnum[name]]}")
        return "\n".join(lines)
