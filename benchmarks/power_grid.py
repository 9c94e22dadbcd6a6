#!/usr/bin/env python
"""Power-delivery grid benchmark: an N x N resistor mesh held by 1 V supply pads (E rows to ground
every `pitch` nodes) with a load current on every node -- the R / A / E netlist the voltage-source
elimination (csrc/sources.cu) exists for.

    python benchmarks/power_grid.py [--n 4096] [--pitch 64] [--reps 3] [--gmres-sizes 512,1024]
                                    [--gmres-maxit 3000] [--out profiles/power_grid.json]

One JSON document (also printed): the card's name and power limit; per rep of the eliminated solve
the split assemble (full MNA CSR), forest, reduce, reduced assembly, AMG setup, solve, expand, the
iterations and relres_full; and the "before": the GMRES path (eliminate_sources=False) on the same
generator at the smaller sizes with an explicit iteration cap -- time, iterations, status, relres.

    python -m torch.distributed.run --nproc-per-node R benchmarks/power_grid.py --distributed [--n ...]

The row-partitioned eliminated solve (Circuit(..., distributed=True), nodal_b200/dist_sources.py)
instead: per rep and per rank the split share upload, full-row exchange and assembly, E gather and
forest, reduction, reduced exchange and assembly, AMG setup and solve (iterations), expansion and
relres_full; rank 0 writes the document."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import nodal_b200 as n  # noqa: E402
from nodal_b200 import generators as gen  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def eliminated(N, pitch, reps):
    net = gen.power_grid(N, pitch, vdd=1.0, load=1e-4, seed=0)
    table = net.table()
    rows = []
    for rep in range(reps + 1):                 # rep 0 warms every kernel and the allocator up
        circuit, asm_ms = timed(lambda: n.Circuit(net, sparse=True))
        sol, total_ms = timed(circuit.solve)
        st = sol.stats
        red = st["reduction"]
        x = sol.result
        src = x[table.kcl:]
        load = float(table.value[table.type == 1].sum())
        row = dict(rep=rep, unknowns=table.n, components=len(table), assemble_ms=asm_ms, solve_total_ms=total_ms,
                   forest_ms=red["forest_ms"], reduce_ms=red["reduce_ms"], reduced_assemble_ms=red["assemble_ms"],
                   amg_setup_ms=st.get("setup_ms"), amg_solve_ms=st.get("solve_ms"),
                   reduced_solve_wall_ms=red["solve_ms"], expand_ms=red["expand_ms"], solver=st["solver"],
                   auto=st.get("auto"), status=st["status"], iterations=st["iterations"], relres_reduced=st["relres"],
                   relres_full=red["relres_full"], reduced_rows=red["reduced_rows"], sources=red["sources"],
                   grounded_nodes=red["grounded_nodes"], forest_depth=red["forest_depth"],
                   source_current_minus_load=float(src.sum() - load) / load,
                   max_potential=float(x[:table.kcl].max()), min_potential=float(x[:table.kcl].min()))
        print(json.dumps(row), flush=True)
        rows.append(row)
        del circuit, sol
    return rows[1:]


def distributed(N, pitch, reps):
    import torch.distributed as dist
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    net = gen.power_grid(N, pitch, vdd=1.0, load=1e-4, seed=0)
    table = net.table()
    rows = []
    for rep in range(reps + 1):                 # rep 0 warms every kernel, the allocator and NCCL up
        dist.barrier()
        circuit, build_ms = timed(lambda: n.Circuit(net, sparse=True, distributed=True))
        sol, total_ms = timed(circuit.solve)
        st, red = sol.stats, sol.stats["reduction"]
        row = dict(rep=rep, rank=rank, world=world, unknowns=table.n, build_ms=build_ms, solve_total_ms=total_ms,
                   upload_ms=red["upload_ms"], full_exchange_assemble_ms=red["full_assemble_ms"],
                   e_gather_forest_ms=red["forest_ms"], reduce_ms=red["reduce_ms"],
                   reduced_exchange_assemble_ms=red["assemble_ms"], amg_setup_ms=st.get("setup_ms"),
                   amg_solve_ms=st.get("solve_ms"), reduced_solve_wall_ms=red["solve_ms"], iterations=st["iterations"],
                   solver=st["solver"], status=st["status"], expand_ms=red["expand_ms"], relres_ms=red["relres_ms"],
                   relres_full=red["relres_full"], reduced_rows=red["reduced_rows"],
                   local_rows=int(circuit.G.shape[0]), local_nnz=circuit.G.nnz)
        if rank == 0:
            print(json.dumps(row), flush=True)
        rows.append(row)
        del circuit, sol
    every = [None] * world
    dist.all_gather_object(every, rows)
    dist.destroy_process_group()
    return rank, [r for per_rank in every for r in per_rank if r["rep"] > 0]


def gmres_before(N, pitch, maxit):
    net = gen.power_grid(N, pitch, vdd=1.0, load=1e-4, seed=0)
    circuit = n.Circuit(net, sparse=True, eliminate_sources=False, maxit=maxit)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        sol, ms = timed(circuit.solve)
    st = sol.stats
    row = dict(n=N, unknowns=net.table().n, solver=st.get("solver"), status=st.get("status"),
               iterations=st.get("iterations"), relres=st.get("relres"), maxit=maxit, ms=ms,
               finite=bool(np.all(np.isfinite(sol.result))), note=st.get("note"))
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--pitch", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gmres-sizes", default="512,1024")
    ap.add_argument("--gmres-maxit", type=int, default=3000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--distributed", action="store_true", help="row-partitioned solve, run under torchrun")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("power_grid.py measures the GPU path: no CUDA device")
    doc = dict(card=card(), n=args.n, pitch=args.pitch, load="uniform [0, 1e-4) A on every node, 1 ohm mesh, 1 V pads")
    if args.distributed:
        rank, doc["distributed"] = distributed(args.n, args.pitch, args.reps)
        doc["world"] = doc["distributed"][0]["world"]
        if rank == 0 and args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                json.dump(doc, fh, indent=1)
        return
    doc["eliminated"] = eliminated(args.n, args.pitch, args.reps)
    doc["gmres_before"] = [gmres_before(int(s), args.pitch, args.gmres_maxit)
                           for s in args.gmres_sizes.split(",") if s]
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])))


if __name__ == "__main__":
    main()
