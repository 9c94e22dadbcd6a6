#!/usr/bin/env python
"""Op-amp stages on a resistive sheet (generators.amplifier_grid): the netlist the Schur-complement
solve (nodal_b200/schur.py, csrc/schur.cu) exists for.

    python benchmarks/amplifier_grid.py [--sizes 1024:128,2048:256] [--reps 2] [--gmres-maxit 3000]
                                        [--ideal-pads] [--pitch P] [--out profiles/amplifier_grid.json]

Each size is N:stages.  One JSON document (also printed): the card's name, power limit and clock;
per size and rep of the Schur solve the split device check, split, AMG setup on L, columns of S
(batches, most iterations of a batch), factor, each refinement step and relres_full; and, on the same
netlist, today's path (schur=False: GMRES(60) with the diagonal preconditioner, capped at
--gmres-maxit iterations) -- status, iterations, relres and wall time.

--ideal-pads: the sheet held by ideal pads (amplifier_grid(..., ideal_pads=True)), solved with
schur=True, eliminate_sources=True (nodal_b200/source_schur.py): per rep the forest, reduced assembly,
split, AMG setup, columns, factor, refinement, expansion and relres_full; and, on the same netlist,
today's schur=True path (the Schur complement of the full system, every pad a row of S) with the
same stages, then GMRES capped at --gmres-maxit where it declines.  --pitch sets the pad pitch (default N // 8),
--rtol / --schur-rtol the tolerances of both."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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


def schur_runs(net, reps, **opts):
    rows = []
    for rep in range(reps + 1):                 # rep 0 warms every kernel and the allocator up
        circuit, asm_ms = timed(lambda: n.Circuit(net, sparse=True, schur=True, **opts))
        sol, total_ms = timed(circuit.solve)
        st = sol.stats["schur"]
        row = dict(rep=rep, assemble_ms=asm_ms, solve_total_ms=total_ms, solver=sol.stats["solver"],
                   status=sol.stats["status"], applied=st["applied"],
                   reason=st.get("reason"), **{k: st.get(k) for k in (
                       "branches", "node_rows", "check_ms", "split_ms", "amg_setup_ms", "batches",
                       "batch_iterations_max", "columns_ms", "factor_ms", "refine_steps", "refine_ms",
                       "refine_iterations", "relres_history", "relres_full")})
        print(json.dumps(row), flush=True)
        rows.append(row)
        del circuit, sol
    return rows[1:]


_SCHUR_KEYS = ("branches", "node_rows", "split_ms", "amg_setup_ms", "batches", "batch_iterations_max", "columns_ms",
               "factor_ms", "refine_steps", "refine_ms", "refine_iterations", "relres_history")


def source_schur_runs(net, reps, **opts):
    rows = []
    for rep in range(reps + 1):                 # rep 0 warms every kernel and the allocator up
        circuit, asm_ms = timed(lambda: n.Circuit(net, sparse=True, schur=True, eliminate_sources=True, **opts))
        sol, total_ms = timed(circuit.solve)
        st = sol.stats
        red, sc = st.get("reduction", {}), st.get("schur", {})
        row = dict(rep=rep, assemble_ms=asm_ms, solve_total_ms=total_ms, solver=st["solver"],
                   reason=red.get("reason"), relres_full=st.get("relres_full"),
                   **{k: red.get(k) for k in ("sources", "supernodes", "reduced_rows", "dependent_rows", "forest_ms",
                                              "reduce_ms", "expand_ms")},
                   reduced_assemble_ms=red.get("assemble_ms"), schur={k: sc.get(k) for k in _SCHUR_KEYS})
        print(json.dumps(row), flush=True)
        rows.append(row)
        del circuit, sol
    return rows[1:]


def todays_path(net, maxit):
    circuit, asm_ms = timed(lambda: n.Circuit(net, sparse=True, maxit=maxit))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sol, ms = timed(circuit.solve)
    st = sol.stats
    row = dict(assemble_ms=asm_ms, solve_ms=ms, solver=st["solver"], status=st["status"],
               iterations=st.get("iterations"), relres=st.get("relres"), note=st.get("note"), maxit=maxit)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", default="1024:128,2048:256")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--gmres-maxit", type=int, default=3000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--ideal-pads", action="store_true")
    ap.add_argument("--pitch", type=int, default=None)
    ap.add_argument("--rtol", type=float, default=1e-10)
    ap.add_argument("--schur-rtol", type=float, default=None, help="tolerance of the L solves (default: --rtol)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("amplifier_grid.py measures the GPU solve: no CUDA device is visible")
    doc = dict(benchmark="amplifier_grid", card=card(), runs=[])
    for item in args.sizes.split(","):
        N, stages = (int(v) for v in item.split(":"))
        net = gen.amplifier_grid(N, stages, seed=args.seed, pitch=args.pitch, ideal_pads=args.ideal_pads)
        t = net.table()
        print(f"# amplifier_grid({N}, {stages}, ideal_pads={args.ideal_pads}): {t.n} unknowns, {t.be} branch rows",
              flush=True)
        run = dict(N=N, stages=stages, pitch=args.pitch or max(1, N // 8), ideal_pads=args.ideal_pads, unknowns=t.n,
                   branches=t.be, components=len(t))
        if args.ideal_pads:
            # today's path declines or misses rtol on these netlists and goes on to GMRES: maxit caps it
            opts = dict(rtol=args.rtol, schur_rtol=args.schur_rtol or args.rtol, maxit=args.gmres_maxit)
            run.update(options=opts, source_schur=source_schur_runs(net, args.reps, **opts),
                       todays_path=schur_runs(net, args.reps, **opts))
        else:
            run.update(schur=schur_runs(net, args.reps), todays_path=todays_path(net, args.gmres_maxit))
        doc["runs"].append(run)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
