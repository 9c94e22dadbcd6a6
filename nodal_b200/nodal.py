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
from . import dist_sources
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
    numpy.linalg.solve).  ``sparse=True``: CSR G, Jacobi-PCG for R/A-only
    netlists, restarted GMRES otherwise (replaces scipy spsolve); R/A/E netlists
    whose voltage sources form a forest are solved through the elimination of
    the sources (``eliminate_sources``, see sources.py); ``schur=True`` solves
    netlists with op-amps and dependent sources through the Schur complement of
    the branch rows (see schur.py), and with ``eliminate_sources=True`` it
    eliminates their voltage sources first (see source_schur.py).

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
        self._schur = schur.check_option(self.options, self.sparse, self.options.get("distributed"))
        table, currents = self.netlist.table_and_currents()
        table.validate()
        self.table = table
        dev = Device.get(self.options.get("device"))
        self._dev = dev
        self._dist = None
        self._dsrc = None
        self._dtab = None
        if self.options.get("distributed"):
            G, A = self._build_distributed(dev, table)
        elif self.sparse:
            # csr_order="first_touch": G's columns in the order the reference's G.tocsr() has before its
            # solve (nodal.py:396-397); the solve then works on the sorted form, as spsolve sorts in place
            order = self.options.get("csr_order", "sorted")
            # tables the source elimination or the Schur solve will take keep their device columns for
            # it (sources.py, schur.py)
            self._eliminate = sources.check_option(self.options, table)
            limit = int(self.options.get("dense_fallback_max_rows", 32768))
            if sources.skip_reason(table, self._eliminate, limit) == "" or self._schur:
                self._dtab = dev.upload_table(table)
            G, A = dev.assemble_csr(table, dtab=self._dtab, order=order)
            if order != "sorted":
                self._G_sorted = dev.assemble_csr(table)[0]
        else:
            G, A = dev.assemble_dense(table, atomic=bool(self.options.get("atomic_stamp", False)))
        logging.debug(f"currents={currents}")
        return [G, A, currents]

    def _build_distributed(self, dev, table):
        """Row-partitioned form (one process per GPU under torchrun, torch.distributed initialised
        with the nccl backend): every rank holds the netlist, uploads the table, selects the
        components touching its rows on the device and builds its rows of G only.  G is then a
        LocalRows view (the rank's rows, global columns), A the rank's slice of the right-hand side."""
        import torch.distributed as tdist
        from . import dist as ndist
        if not self.sparse:
            raise ValueError("distributed=True needs sparse=True (the dense LU is single-GPU)")
        if not (tdist.is_available() and tdist.is_initialized()):
            raise RuntimeError("distributed=True needs an initialised torch.distributed process group")
        rank, world = tdist.get_rank(), tdist.get_world_size()
        if dist_sources.applies(table):
            # R / A / E netlists: through the row-partitioned elimination of the sources (dist_sources.py)
            self._dsrc = dist_sources.DistSources(self, dev, table, rank, world)
            return self._dsrc.G, self._dsrc.A
        runner = ndist.GridRunner(dev, table, 0, rank, world, rtol=self.options.get("rtol", 1e-10),
                                  precond="jacobi" if self.options.get("precond") == "jacobi" else "amg",
                                  amg=self.options.get("amg"), solver=ndist.shared_solver(dev, rank, world))
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
    def _sparse_solver(self):
        """Which device solver the sparse path uses: "amg", "pcg" or "gmres".
        precond: "auto" (default) = aggregation-AMG preconditioned CG for R / A netlists, with a
        Jacobi-PCG retry if the hierarchy cannot be built or the solve does not converge (the
        behaviour on singular systems is then the Jacobi path's); "amg" / "jacobi" force one."""
        precond = self.options.get("precond", "auto")
        if precond not in ("auto", "jacobi", "amg"):
            raise ValueError(f"precond must be 'auto', 'jacobi' or 'amg', got {precond!r}")
        if not self.table.is_spd_structured():
            return "gmres"
        return "pcg" if precond == "jacobi" else "amg"

    def _device_solve(self, rhs, amg=None):
        """x, info for G x = rhs on the device (rhs is a device tensor; dense G is not modified).
        Distributed circuits: rhs and x are the rank's slices."""
        dev = self._dev
        if not self.sparse:
            return dev.lu_solve(self.G.clone(), rhs)
        if self._dsrc is not None:
            raise NotImplementedError("the row-partitioned solve of a netlist with voltage sources is implemented "
                                      "for solve() only")
        kind = self._sparse_solver()
        rtol = self.options.get("rtol", 1e-10)
        warm = self._warm_start()
        if getattr(self, "_G_sorted", None) is not None:
            self.G = self._G_sorted        # spsolve leaves circuit.G with sorted indices too (SURVEY.md app. C-5)
            self._G_sorted = None
        if self._dist is not None:
            if kind == "gmres":
                raise NotImplementedError("row-partitioned solve is implemented for R / A netlists")
            g, run = self.G, self._dist
            first = None
            if kind == "amg":
                x, info = run.pcg.solve_amg(g.n, g.bounds, g.indptr, g.indices, g.data, rhs, rtol=rtol,
                                            maxit=self.options.get("maxit"), **(self.options.get("amg") or {}))
                if info["status"] == 0 or self.options.get("precond") == "amg":
                    return x, info
                first = f"dist_amg_pcg status {info['status']}"      # same status on every rank
            x, info = run.pcg.solve(g.n, g.bounds, g.indptr, g.indices, g.data, rhs, rtol=rtol,
                                    maxit=self.options.get("maxit"))
            if first:
                info["fallback_from_amg"] = first
            return x, info
        if kind in ("amg", "pcg"):
            return self._spd_solve(self.G, rhs, kind, rtol, warm, amg)
        x, info = dev.gmres(self.G, rhs, rtol=self.options.get("rtol", 1e-12),
                            restart=self.options.get("restart", 60),
                            maxit=self.options.get("maxit") or 20000)
        # The reference's sparse path is a direct solve, exact for any non-singular MNA system; the
        # diagonally preconditioned GMRES can stall on indefinite systems with many source /
        # op-amp rows.  Rather than handing back an unconverged iterate, systems that fit the dense
        # LU go through it; larger ones are reported (NaNs + warning in solve(), as for breakdown).
        if info["status"] == 2 and self.options.get("gmres_fallback", True):
            limit = int(self.options.get("dense_fallback_max_rows", 32768))
            if self.G.n <= limit:
                x, lu = dev.lu_solve(dev.csr_to_dense(self.G), rhs)
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
        dev = self._dev
        if kind == "amg" and amg is None and warm is None and self.options.get("precond", "auto") == "auto":
            # "auto": which preconditioner pays depends on the graph, not on its size -- on a 4 M-node
            # expander-like random network Jacobi-PCG needs 98 iterations (43 ms) and the AMG hierarchy
            # 265 ms; on a banded random network of the same size it is 4 616 iterations (1.9 s)
            # against 68 (156 ms); grids are the second kind.  A short Jacobi-PCG probe tells them
            # apart: if 24 iterations gained two digits it will finish in ~100, otherwise its iterate
            # is the initial guess of the AMG solve.
            probe_its = int(self.options.get("auto_probe_iterations", 24))
            if G.n >= self.options.get("auto_probe_min_rows", 50_000) and probe_its > 0:
                x0, info0 = dev.pcg(G, rhs, rtol=rtol, maxit=probe_its, flags=self.options.get("pcg_flags", 0))
                if info0["status"] == 0:
                    info0["auto"] = "jacobi (converged inside the probe)"
                    return x0, info0
                if info0["status"] == 2 and info0["relres"] <= 1e-2:
                    x, info = dev.pcg(G, rhs, rtol=rtol, maxit=self.options.get("maxit"), x0=x0,
                                      flags=self.options.get("pcg_flags", 0))
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
        return dev.pcg(G, rhs, rtol=rtol, maxit=self.options.get("maxit"),
                      flags=self.options.get("pcg_flags", 0), x0=warm)

    def _warm_start(self):
        """Initial guess of the iterative solvers: Circuit(..., x0=array of n values) -- e.g. the
        previous solution of a parameter sweep (SURVEY.md section 5).  None: start from zero."""
        x0 = self.options.get("x0")
        if x0 is None or not self.sparse or self._dist is not None:
            return None
        arr = np.ascontiguousarray(x0, dtype=np.float64)
        if arr.shape != (self.table.n,):
            raise ValueError(f"x0 must have {self.table.n} entries")
        return self._dev.to_device(arr)

    def _amg_solve(self, G, rhs, amg, rtol, x0):
        """AMG-preconditioned CG on one GPU; Jacobi-PCG retry unless precond="amg" was forced."""
        dev = self._dev
        from . import _lib
        try:
            if amg is not None:
                x, info = amg.solve(rhs, rtol=rtol, maxit=self.options.get("maxit"), x0=x0)
            elif G.n >= self.options.get("amg_graph_min_rows", 100_000):
                # large systems: the graph-captured form (csrc/dist_amg.cu with one rank):
                # one CUDA graph per iteration, no host round trip inside the iteration
                from . import dist as ndist
                g = G
                bounds = np.array([0, g.n], dtype=np.int32)
                x, info = ndist.single_solver(dev).solve_amg(
                    g.n, bounds, g.indptr, g.indices, g.data, rhs, rtol=rtol, maxit=self.options.get("maxit"),
                    x0=x0, **(self.options.get("amg") or {}))
            else:
                x, info = dev.amg_pcg(G, rhs, rtol=rtol, maxit=self.options.get("maxit"), x0=x0,
                                      **(self.options.get("amg") or {}))
            if info["status"] == 0 or self.options.get("precond") == "amg":
                return x, info
            first = f"amg_pcg status {info['status']} after {info['iterations']} iterations"
        except _lib.NodalLibraryError as err:
            if self.options.get("precond") == "amg":
                raise
            first = str(err)
        x, info = dev.pcg(G, rhs, rtol=rtol, maxit=self.options.get("maxit"),
                          flags=self.options.get("pcg_flags", 0))
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
        UnconnectedCircuitError like the dense path."""
        if self.sparse and self.options.get("check_connected") and not self.is_connected():
            logging.error("Model error: unconnected circuit")
            raise UnconnectedCircuitError
        # R / A / E netlists: through the elimination of the voltage sources when it applies
        # (sources.py; dist_sources.py row-partitioned, x whole on every rank); otherwise `info` is
        # the stats of why not, or None
        if self._dsrc is not None:
            x, info = self._dsrc.solve()
        else:
            x, info = sources.solve(self) if self.sparse and self._dist is None else (None, None)
        if x is None:
            skipped = info
            # schur=True with eliminate_sources=True on a table with E rows and dependent rows: the
            # elimination, then the Schur complement of the reduced system (source_schur.py)
            x, info = source_schur.solve(self) if self.sparse and self._dist is None else (None, None)
            if x is not None:
                skipped = None
            elif info is not None:
                skipped = info
        if x is None:
            # then, when requested and the netlist qualifies, the Schur complement of the branch rows
            x, info = schur.solve(self) if self.sparse and self._dist is None else (None, None)
            if x is None:
                declined = info
                x, info = self._device_solve(self.A)
                if declined is not None:
                    info["schur"] = declined
            if skipped is not None:
                info["reduction"] = skipped
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
        if self.sparse and run is None and self._sparse_solver() == "amg" and len(pairs) > 1:
            from . import _lib
            try:
                amg = dev.amg(self.G, **(self.options.get("amg") or {}))
            except _lib.NodalLibraryError:
                if self.options.get("precond") == "amg":
                    raise
                amg = None             # _device_solve retries per right-hand side and falls back to Jacobi
        values, stats = [], []
        try:
            if amg is not None and self.options.get("multi_rhs", True):
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
                    xs, infos = amg.solve_multi(rhs, rtol=self.options.get("rtol", 1e-10), maxit=self.options.get("maxit"))
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
