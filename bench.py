#!/usr/bin/env python
"""Headline benchmark: equivalent-resistance solve of a 16M-node resistor grid (config C5a).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--grid 4096]
                    [--precond amg|jacobi] [--dump-outputs DIR]

One "step" is one pass of the hot path over the workload: (N > 1: select the rank's components
on the device ->) stamp the component table -> build the CSR -> AMG-preconditioned CG (default;
--precond jacobi = the round-1 headline) to relres 1e-10 -> R = e(1) - e(g).  The same algorithm
runs on every GPU count (rows partitioned over the ranks).
  value : unknowns / s with the component table already resident in HBM
  e2e   : the same through the public API with HOST buffers (pinned table H2D and the whole
          solution vector D2H inside the timed region, on every rank)
  roofline : the level-0 SELL sweep of the AMG cycle (Jacobi: the PCG's SpMV + dot kernel),
          per-launch time from CUDA events, algorithmic bytes in DESIGN.md
  cpu_baseline : the unmodified reference (baseline/_ref; oracle port if absent) on a bounded
          sample of the same workload; same_size_pair: that sample through this repo as well
Prints ONE JSON line on rank 0.

--dump-outputs DIR writes, after the timed steps, what the last timed step computed as float64 .npy files,
so that two builds can be compared output for output (the workload is deterministic for given arguments):
  R                       e(1) - e(g) of the value leg
  potentials_sample       the solved node potentials at a fixed, seeded sample of 2^20 rows (all rows of
                          a smaller system): the whole vector of the 4096 grid would be 134 MB
  potentials_sample_rows  the row index of each sampled potential
  R_e2e                   R of the e2e leg (public API)
--impl reference writes R only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"     # keep NCCL's version banner off stdout (one JSON line only)

import numpy as np  # noqa: E402

RTOL = 1e-10
# DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full) of the roofline kernels,
# read from the committed capture summaries: profiles/ncu_traffic.json = {kernel: {grid side: bytes, "source": csv}}
def ncu_traffic(kernel, N):
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            entry = json.load(fh).get(kernel, {})
        return entry.get(str(N))
    except (OSError, ValueError):
        return None


KNIGHT_LIMIT = 4 / np.pi - 0.5       # infinite-grid knight's-move resistance
DUMP_ROWS = 1 << 20                  # potentials written by --dump-outputs: 8 MB, plus 8 MB of row indices


def sample_rows(n):
    """The sorted rows of the solution that --dump-outputs writes: a fixed, seeded sample."""
    if n <= DUMP_ROWS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def gather_rows(x_local, row0, rows, world):
    """x[rows] of a solution of which this rank holds rows row0 .. row0 + len(x_local), on every rank."""
    import torch
    idx = torch.from_numpy(rows).to(x_local.device)
    mine = (idx >= row0) & (idx < row0 + x_local.numel())
    out = torch.zeros(len(rows), dtype=torch.float64, device=x_local.device)
    out[mine] = x_local[idx[mine] - row0]
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(out)                 # each row has one owner; the other ranks add exact zeros
    return out.cpu().numpy()


def write_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.asarray(a, dtype=np.float64))


# --------------------------------------------------------------------------- reference arm
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def grid_rows(N):
    """csv rows of the N x N 1-ohm grid of SURVEY.md section 8(d) (config C2 / C5a): for every site in row-major
    order one resistor to the (x+1, y) and one to the (x, y+1) neighbour; probe node "1" at (N//2, N//2),
    ground "g" a knight's move away at (N//2+2, N//2+1)."""
    def name(x, y):
        if (x, y) == (N // 2, N // 2):
            return "1"
        if (x, y) == (N // 2 + 2, N // 2 + 1):
            return "g"
        return f"n{x}_{y}"
    rows = []
    for x in range(N):
        for y in range(N):
            if x + 1 < N:
                rows.append([f"r{len(rows)}", "R", "1.0", name(x, y), name(x + 1, y)])
            if y + 1 < N:
                rows.append([f"r{len(rows)}", "R", "1.0", name(x, y), name(x, y + 1)])
    return rows


def grid_csv(N):
    """The N x N grid netlist as the csv FILE the reference reads (written outside any timed region)."""
    import csv
    import tempfile
    fd, path = tempfile.mkstemp(prefix=f"grid{N}_", suffix=".csv")
    with os.fdopen(fd, "w", newline="") as fh:
        csv.writer(fh).writerows(grid_rows(N))
    return path


def reference_available():
    return os.path.isfile(os.path.join(REF_DIR, "nodal", "nodal.py"))


def reference_step(N, path=None):
    """One pass of the hot path on the host CPU over an N x N grid: csv file -> Netlist ->
    equivalent_resistance(..., sparse=True) (numbering, deepcopy, per-item DOK stamping, spsolve).
    Runs the UNMODIFIED reference from baseline/_ref (baseline/install_ref.py) when it is there
    (kind "reference"), else the oracle port of the same algorithm (kind "port").
    Returns (seconds, unknowns, R, kind)."""
    own = path is None
    if own:
        path = grid_csv(N)
    try:
        if reference_available():
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)
            import logging
            import nodal as ref                      # the reference package, not this repo's
            import nodal.equiv
            logging.getLogger().setLevel(logging.ERROR)
            t0 = time.perf_counter()
            net = ref.Netlist(path)
            r = ref.equiv.equivalent_resistance(net, "1", "g", sparse=True)
            dt = time.perf_counter() - t0
            return dt, N * N - 1, float(r), "reference"
        from oracle import mna_oracle as orc
        import csv
        t0 = time.perf_counter()
        with open(path) as fh:
            rows = [row for row in csv.reader(fh, skipinitialspace=True)]
        r = orc.equivalent_resistance(rows, "1", "g", sparse=True, backend="dok")
        dt = time.perf_counter() - t0
        return dt, N * N - 1, float(r), "port"
    finally:
        if own:
            os.unlink(path)


def cpu_baseline_entry(N, dt, unknowns, r, kind, full_grid):
    what = ("the unmodified reference package (baseline/_ref): Netlist(csv) + equivalent_resistance(sparse=True)"
            if kind == "reference" else
            "oracle port of the reference algorithm (csv rows -> numbering -> per-item scipy DOK stamping -> spsolve)")
    return {"value": unknowns / dt, "unit": "unknowns/s", "cores": 1, "kind": kind,
            "sample": f"{N}x{N} grid ({unknowns} unknowns) through {what} in {dt:.1f} s, R={r!r}; single-threaded "
                      f"by construction (Python stamping loop + SuperLU); the full {full_grid}x{full_grid} workload "
                      f"cannot run on this path (SuperLU MemoryError, BASELINE.md 2.2)",
            "host_cpus": os.cpu_count(), "seconds": dt, "grid": N}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N = args.ref_grid
    small = grid_csv(max(20, N // 8))
    path = grid_csv(N)
    try:
        for _ in range(args.warmup):
            reference_step(max(20, N // 8), small)
        times = []
        for _ in range(args.steps):
            dt, unknowns, r, kind = reference_step(N, path)
            times.append(dt)
    finally:
        os.unlink(small)
        os.unlink(path)
    total = sum(times)
    value = args.steps * unknowns / total
    line = {
        "impl": "reference", "metric": "unknowns_per_second", "value": value, "unit": "unknowns/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"grid2d_{args.grid}x{args.grid} equivalent resistance (config C5a)",
                   "sample": f"grid2d_{N}x{N}", "warmup_sample": f"grid2d_{max(20, N // 8)}"},
        "cpu_baseline": cpu_baseline_entry(N, total / args.steps, unknowns, r, kind, args.grid),
        "e2e": {"value": value, "unit": "unknowns/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cpus": os.cpu_count(), "R": r,
    }
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"R": [r]})
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "samples": len(sm),
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- our arm
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_ours(args):
    import torch
    import torch.distributed as dist
    import nodal_b200 as n
    from nodal_b200 import _lib
    from nodal_b200 import dist as ndist
    from nodal_b200 import generators as gen
    from nodal_b200.device import Device

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = Device.get(local)
    lib = dev.lib
    N = args.grid
    precond = args.precond
    amg_opts = {"gather_below": args.gather_below} if args.gather_below else {}

    # ---- workload (host, untimed): grid netlist + the 1 A probe source of equivalent_resistance
    import copy
    net = gen.grid2d(N)
    probe = copy.deepcopy(net)
    probe.process_component(["a1", "A", "1", "1", "g"])      # equiv.py:51
    table = probe.table()
    table.facts()                                             # the host scan of the columns (cached with the table)
    n_unknowns, ncomp = table.n, len(table)
    row_1 = probe.nodenum["1"]

    # value leg: the whole component table resident in HBM on every rank; one step = (N > 1: select the
    # rank's components on the device) + stamp + CSR build of the rank's rows + partitioned solve + R
    classic_jacobi = world == 1 and precond == "jacobi"      # the tuned single-GPU Jacobi-PCG of round 1
    runner = None
    if not classic_jacobi:
        runner = ndist.GridRunner(dev, table, row_1, rank, world, rtol=RTOL, precond=precond, amg=amg_opts,
                                  solver=ndist.shared_solver(dev, rank, world) if world > 1 else ndist.single_solver(dev))
    dtab = dev.upload_table(table)
    torch.cuda.synchronize()

    def step_device():
        """(R, info, the rank's rows of the solution)"""
        if runner is not None:
            r, info = runner.step(dtab)
            return r, info, runner.x_local
        csr, rhs = dev.assemble_csr(table, dtab=dtab)
        x, info = dev.pcg(csr, rhs, rtol=RTOL)
        info["nnz"] = csr.nnz
        return float(x[row_1]), info, x                       # e(1) - e(g), ground is 0 V

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        r, info, x_local = step_device()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = lib.nodal_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    iters, infos = [], []
    for _ in range(args.steps):
        r, info, x_local = step_device()
        iters.append(info["iterations"])
        infos.append(info)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.nodal_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        rows = sample_rows(n_unknowns)
        row0 = int(runner.bounds[rank]) if runner is not None else 0
        dump = {"R": [r], "potentials_sample": gather_rows(x_local, row0, rows, world),
                "potentials_sample_rows": rows}
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = n_unknowns / (ms_per_step * 1e-3)
    nnz = info["nnz"]

    # ---- e2e leg: the public API with HOST buffers.  Every rank holds the netlist (pinned columns);
    # equivalent_resistance(netlist, "1", "g", sparse=True[, distributed=True]) -- the call behind
    # `nodal-resistance FILE -s` (nodal/equiv.py:31-61) -- uploads the table, (selects the rank's
    # components on the device,) assembles, solves and reads the two probe potentials back.
    import nodal_b200.equiv
    net.table().pin_memory()
    net.table().facts()
    opts = dict(rtol=RTOL, precond=precond)
    if world > 1:
        opts["distributed"] = True
    if amg_opts and precond != "jacobi":
        opts["amg"] = amg_opts

    def step_e2e():
        r_ = n.equiv.equivalent_resistance(net, "1", "g", sparse=True, **opts)
        return float(r_), n.equiv.equivalent_resistance.last_stats

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        r_e2e, e2e_stats = step_e2e()
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    e2e_ms = max(ev0.elapsed_time(ev1), wall * 1e3)
    if world > 1:
        t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_ms /= args.steps
    e2e = {"value": n_unknowns / (e2e_ms * 1e-3), "unit": "unknowns/s",
           "h2d_bytes_per_step": int(Device.uploaded_bytes(net.table())), "d2h_bytes_per_step": 16 * world,
           "ms_per_step": e2e_ms, "R": r_e2e, "solver": e2e_stats.get("solver"),
           "api": "nodal_b200.equiv.equivalent_resistance(netlist, '1', 'g', sparse=True" +
                  (", distributed=True" if world > 1 else "") + ") on a host TableNetlist (pinned columns) on every "
                  "rank: every rank uploads its 1/N share of the table (the rows a rank stamps reach it over NVLink), "
                  "the two probe potentials come down (bytes summed over ranks)"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump["R_e2e"] = [r_e2e]
        write_outputs(args.dump_outputs, dump)

    # ---- roofline of the dominant kernel, per-launch time from CUDA events (rank 0, one GPU's share)
    peak, peak_src = load_peaks()
    roof, amg_side, jac_side = None, None, None
    if world == 1:
        csr, rhs = dev.assemble_csr(table, dtab=dtab)
        if precond == "jacobi":
            _, prof = dev.pcg(csr, rhs, rtol=RTOL, maxit=256, flags=_lib.PCG_PROFILE)
            km = prof.get("kernel_ms")
            if km:
                bytes_spmv = 12.0 * nnz + 20.0 * n_unknowns
                achieved = bytes_spmv / (km["spmv_dot"] * 1e-3) / 1e9
                roof = {"bound": "hbm", "kernel": "pcg_spmv_dot_sell_kernel", "achieved": achieved, "peak": peak,
                        "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                        "traffic": ncu_traffic("pcg_spmv_dot_sell_kernel", N),
                        "algorithmic_bytes_per_launch": bytes_spmv, "ms_per_launch": km["spmv_dot"],
                        "samples": km["samples"],
                        "other_kernels_ms": {"update": km["update"], "direction": km["direction"]},
                        "frac_of_nominal_8TBs": achieved / 8000.0}
        else:
            # level-0 SELL sweeps of the AMG-PCG step: 3 per iteration (CG q = A p, residual of the pre-smoothed
            # iterate, post-smoothing sweep).  Algorithmic bytes: 12 nnz (value + column) + per row the gathered
            # vector once (8), the right-hand side (8), the diagonal (8, Jacobi sweep only) and the result (8).
            h = dev.amg(csr)
            km = h.profile_sweeps(reps=64)
            h.close()
            by = {"jacobi": 12.0 * nnz + 32.0 * n_unknowns, "residual": 12.0 * nnz + 24.0 * n_unknowns,
                  "spmv_dot": 12.0 * nnz + 16.0 * n_unknowns}
            achieved = by["jacobi"] / (km["jacobi"] * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "amg_sell_kernel<2> (level-0 damped-Jacobi sweep)", "achieved": achieved,
                    "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                    "traffic": ncu_traffic("amg_sell_kernel<2>", N),
                    "algorithmic_bytes_per_launch": by["jacobi"], "ms_per_launch": km["jacobi"], "samples": 64,
                    "other_kernels_ms": {"level0_residual_sweep": km["residual"], "level0_spmv_dot": km["spmv_dot"]},
                    "other_kernels_gbs": {"level0_residual_sweep": by["residual"] / km["residual"] / 1e6,
                                          "level0_spmv_dot": by["spmv_dot"] / km["spmv_dot"] / 1e6},
                    "frac_of_nominal_8TBs": achieved / 8000.0}
        # ---- the other preconditioner on the same system, beside the headline (one warm-up + one timed step)
        if not args.no_side:
            try:
                for _ in range(2):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    csr, rhs = dev.assemble_csr(table, dtab=dtab)
                    xa, ia = (dev.pcg(csr, rhs, rtol=RTOL) if precond != "jacobi" else dev.amg_pcg(csr, rhs, rtol=RTOL))
                    ra = float(xa[row_1])
                    torch.cuda.synchronize()
                    wall = (time.perf_counter() - t0) * 1e3
                side = {"ms_per_step": wall, "setup_ms": ia["setup_ms"], "solve_ms": ia["solve_ms"],
                        "iterations": ia["iterations"], "relres": ia["relres"], "status": ia["status"], "R": ra,
                        "R_rel_diff_vs_headline": abs(ra - r) / abs(r)}
                if precond != "jacobi":
                    side["pcg_achieved_gbs"] = (12.0 * nnz + 108.0 * n_unknowns) * ia["iterations"] / ia["solve_ms"] / 1e6
                    jac_side = side
                else:
                    side.update(levels=ia["level_rows"], operator_complexity=ia["operator_complexity"])
                    amg_side = side
            except Exception as exc:      # the headline line must not depend on the side measurement
                amg_side = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only), and the SAME sample through this
    # repo from the same csv file with the same call sequence (file -> netlist -> equivalent_resistance):
    # a like-for-like pair next to the headline, whose CPU arm cannot run the full size
    cpu, same = None, None
    if world == 1 and not args.no_cpu_baseline:
        from nodal_b200 import cli
        import nodal_b200.equiv
        Ns = args.ref_grid
        path = grid_csv(Ns)
        try:
            def gpu_from_csv():
                netl = cli.load_netlist_or_exit(path)         # what nodal-resistance FILE -s does
                return float(n.equiv.equivalent_resistance(netl, "1", "g", sparse=True))
            gpu_from_csv()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r_gpu = gpu_from_csv()
            torch.cuda.synchronize()
            t_gpu = time.perf_counter() - t0
            dt, unk, r_cpu, kind = reference_step(Ns, path)
        finally:
            os.unlink(path)
        cpu = cpu_baseline_entry(Ns, dt, unk, r_cpu, kind, N)
        same = {"grid": Ns, "unknowns": unk, "what": "csv file -> netlist -> equivalent_resistance(sparse=True), "
                "host numbering / ingest included on both sides", "gpu_s": t_gpu, "cpu_s": dt, "cpu_kind": kind,
                "speedup": dt / t_gpu, "R_gpu": r_gpu, "R_cpu": r_cpu, "R_rel_diff": abs(r_gpu - r_cpu) / abs(r_cpu)}

    solver_name = {"amg": "aggregation-AMG preconditioned CG", "jacobi": "Jacobi-PCG"}[precond]
    keys = ("assemble_wall_ms", "solve_wall_ms", "setup_ms", "solve_ms", "host_ms", "comm", "levels", "distributed_levels",
            "level_rows", "replicated_rows", "kernels_per_iteration", "halo_recv", "restarts")
    line = {
        "metric": "unknowns_per_second", "value": value, "unit": "unknowns/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"grid2d_{N}x{N} equivalent resistance (config C5a): "
                               f"{'select rank rows + ' if world > 1 else ''}stamp + CSR build + {solver_name} rtol {RTOL}",
                   "unknowns": n_unknowns, "components": ncomp, "nnz": nnz, "precond": precond,
                   "l2": "working set (>= 1.3 GB per level-0 sweep) is larger than the 126 MB L2",
                   "parallelism": f"rows x{world}" if world > 1 else "single GPU"},
        "time_to_solution_s": ms_per_step * 1e-3, "iterations": iters, "relres": info["relres"],
        "R": r, "R_minus_infinite_grid_limit": r - KNIGHT_LIMIT,
        "step_breakdown": {k: info[k] for k in keys if k in info},
        "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "roofline": roof,
        "cpu_baseline": cpu, "same_size_pair": same,
        "jacobi_pcg_side": jac_side, "amg_pcg_side": amg_side,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=4096, help="grid side (4096 -> 16.7M nodes, config C5a)")
    ap.add_argument("--ref-grid", type=int, default=400, help="grid side of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precond", default="amg", choices=["amg", "jacobi"],
                    help="preconditioner of the timed step on every GPU count (jacobi: the round-1 headline)")
    ap.add_argument("--gather-below", type=int, default=0,
                    help="AMG: levels with at most this many rows are replicated on every rank (0 = library default)")
    ap.add_argument("--no-side", action="store_true", help="skip the side measurement of the other preconditioner")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
