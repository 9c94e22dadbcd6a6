#!/usr/bin/env python
"""Per-launch time of the level-0 kernels of the AMG V-cycle on the headline system (the N x N grid
of bench.py with its 1 A probe source), in the unfused form (Jacobi start, residual sweep,
prolongation, damped-Jacobi sweep) and the fused form (amg_cycle_sweep_kernel MODE 1 and 2).

    python benchmarks/amg_cycle.py [--n 4096] [--reps 64] [--out profiles/amg_cycle.json]

Times come from CUDA events around `reps` back-to-back launches of each kernel on the hierarchy's
own level-0 operator, aggregates and work vectors (csrc/amg.cu, nodal_amg_profile_cycle); the
working set is far larger than the L2.  Bytes are the algorithmic ones: 12 per stored entry (value +
column) plus every vector read or written once per row (gathered vectors counted once: neighbouring
rows reuse them from the cache).  One JSON document (also printed), with the card's name and power
limit."""
import argparse
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from nodal_b200 import generators as gen  # noqa: E402
from nodal_b200.device import Device  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def algorithmic_bytes(n, nnz, nc):
    return {
        "jacobi0": 24.0 * n,                            # b, d^-1 read; x0 written
        "residual": 12.0 * nnz + 24.0 * n,              # x0 gathered, b read, r written
        "prolong": 20.0 * n + 8.0 * nc,                 # x0, agg read, xc gathered, x~ written
        "jacobi": 12.0 * nnz + 32.0 * n,                # x~ gathered, b, d^-1 read, y written
        "fused_residual": 12.0 * nnz + 24.0 * n,        # b, d^-1 gathered, r written
        "fused_post": 12.0 * nnz + 28.0 * n + 8.0 * nc,  # b, d^-1, agg gathered, xc gathered, y written
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 64:
        ap.error("--reps must be at least 64")
    if not torch.cuda.is_available():
        sys.exit("amg_cycle.py needs a CUDA device")
    dev = Device.get(0)
    net = copy.deepcopy(gen.grid2d(args.n))
    net.process_component(["a1", "A", "1", "1", "g"])
    csr, _ = dev.assemble_csr(net.table())
    h = dev.amg(csr)
    try:
        ms = h.profile_cycle(reps=args.reps)
        rows, nnz = list(h.rows), list(h.nnz)
    finally:
        h.close()
    n, nc = rows[0], rows[1]
    by = algorithmic_bytes(n, nnz[0], nc)
    kernels = {k: {"ms_per_launch": ms[k], "algorithmic_bytes": by[k], "gb_per_s": by[k] / (ms[k] * 1e-3) / 1e9}
               for k in ms}
    pairs = {
        "residual": {"unfused_ms": ms["jacobi0"] + ms["residual"], "fused_ms": ms["fused_residual"],
                     "unfused_bytes": by["jacobi0"] + by["residual"], "fused_bytes": by["fused_residual"]},
        "post_smoothing": {"unfused_ms": ms["prolong"] + ms["jacobi"], "fused_ms": ms["fused_post"],
                           "unfused_bytes": by["prolong"] + by["jacobi"], "fused_bytes": by["fused_post"]},
    }
    for p in pairs.values():
        p["saved_ms"] = p["unfused_ms"] - p["fused_ms"]
    doc = {"card": card(), "system": f"grid2d_{args.n}x{args.n} + 1 A probe", "level0_rows": n, "level0_nnz": nnz[0],
           "level1_rows": nc, "reps": args.reps, "kernels": kernels, "pairs": pairs}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
