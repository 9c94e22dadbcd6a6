#!/usr/bin/env python
"""Per-launch time of the level-0 kernels of the AMG V-cycle on the headline system (the N x N grid
of bench.py with its 1 A probe source), in the unfused form (Jacobi start, residual sweep,
prolongation, damped-Jacobi sweep) and the fused form (amg_cycle_sweep_kernel MODE 1 and 2), plus the
fused sweeps and the operator product `spmv_dot` with the operator stored in each SELL entry encoding
(`spmv_dot` is amg_sell_kernel<0>, y = A x with per-block partials of x.y, as nodal_amg_profile_sweeps
times it; it stands in for the CG's acg_spmv_dots_kernel, which has the same row product): compact (the encoding the library picks for this grid) and wide (NODAL_SELL_WIDE=1),
both hierarchies built in the same process.

    python benchmarks/amg_cycle.py [--n 4096] [--reps 64] [--out profiles/amg_cycle.json]

Times come from CUDA events around `reps` back-to-back launches of each kernel on the hierarchy's
own level-0 operator, aggregates and work vectors (csrc/amg.cu, nodal_amg_profile_cycle); the
working set is far larger than the L2.  Bytes are the algorithmic ones: 12 per stored entry (value +
column) wide, 3 compact (column offset + value index), plus every vector read or written once per row
(gathered vectors counted once: neighbouring rows reuse them from the cache).  One JSON document (also printed), with the card's name and power
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


def algorithmic_bytes(n, nnz, nc, entry=12.0):
    """entry: bytes per stored entry, 12 (wide) or 3 (compact)."""
    return {
        "jacobi0": 24.0 * n,                               # b, d^-1 read; x0 written
        "residual": entry * nnz + 24.0 * n,                # x0 gathered, b read, r written
        "prolong": 20.0 * n + 8.0 * nc,                    # x0, agg read, xc gathered, x~ written
        "jacobi": entry * nnz + 32.0 * n,                  # x~ gathered, b, d^-1 read, y written
        "fused_residual": entry * nnz + 24.0 * n,          # b, d^-1 gathered, r written
        "fused_post": entry * nnz + 28.0 * n + 8.0 * nc,   # b, d^-1, agg gathered, xc gathered, y written
        "spmv_dot": entry * nnz + 16.0 * n,                # amg_sell_kernel<0>: x gathered and read, y written
    }


def encoding_rows(dev, csr, reps):
    """Per-launch time of the level-0 fused sweeps and spmv_dot with the operator compact and wide."""
    out = {}
    for name, wide in (("compact", False), ("wide", True)):
        if wide:
            os.environ["NODAL_SELL_WIDE"] = "1"
        try:
            h = dev.amg(csr)
        finally:
            os.environ.pop("NODAL_SELL_WIDE", None)
        try:
            ms = h.profile_cycle(reps=reps)
            ms["spmv_dot"] = h.profile_sweeps(reps=reps)["spmv_dot"]
            n, nnz, nc = h.rows[0], h.nnz[0], h.rows[1]
        finally:
            h.close()
        by = algorithmic_bytes(n, nnz, nc, 12.0 if wide else 3.0)
        out[name] = {k: {"ms_per_launch": ms[k], "algorithmic_bytes": by[k], "gb_per_s": by[k] / (ms[k] * 1e-3) / 1e9}
                     for k in ("fused_residual", "fused_post", "spmv_dot")}
    for k in out["wide"]:
        out.setdefault("compact_over_wide", {})[k] = out["compact"][k]["ms_per_launch"] / out["wide"][k]["ms_per_launch"]
    return out


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
    os.environ["NODAL_SELL_WIDE"] = "1"     # the unfused/fused comparison as recorded before compact entries
    try:
        h = dev.amg(csr)
    finally:
        os.environ.pop("NODAL_SELL_WIDE", None)
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
           "level1_rows": nc, "reps": args.reps, "kernels": kernels, "pairs": pairs,
           "encodings": encoding_rows(dev, csr, args.reps)}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
