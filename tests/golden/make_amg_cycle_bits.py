#!/usr/bin/env python
"""Record the exact bits the AMG V-cycle computes, for tests/test_gpu_amg_cycle_bits.py.

Usage (on a GPU, with the library built from the tree whose results are the reference):
    python tests/golden/make_amg_cycle_bits.py [out.json]

Writes tests/golden/amg_cycle_bits.json (or `out.json`): the SHA-256 of the float64 bytes, and a
few leading values for diagnosis, of
  * amg.apply(r) on the grid40, grid96 and random systems of tests/test_gpu_amg.py (same seeds),
    the single-GPU cycle (csrc/amg.cu);
  * the solution and iteration count of DistPCG.solve_amg with one rank on the 400 x 400 grid
    with gather_below=5000, so several levels take the row-partitioned cycle (csrc/dist_amg.cu).
A change to the cycle's kernels that keeps every rounding step must leave all of them unchanged.
"""
import copy
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

APPLY_CASES = ("grid40", "grid96", "random")
DIST_GRID = 400
DIST_GATHER_BELOW = 5000


def digest(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(), "n": int(a.size), "head": [float(v) for v in a[:4]]}


def apply_bits(device, name):
    from test_gpu_amg import cases
    from test_gpu_sparse import to_device_csr
    A, _ = cases(name)
    r = np.random.default_rng(5).standard_normal(A.shape[0])
    amg = device.amg(to_device_csr(device, A))
    try:
        z = amg.apply(device.to_device(r)).cpu().numpy()
    finally:
        amg.close()
    return z


def dist_bits(device):
    from nodal_b200 import dist as ndist
    from nodal_b200 import generators as gen
    net = copy.deepcopy(gen.grid2d(DIST_GRID))
    net.process_component(["a1", "A", "1", "1", "g"])
    table = net.table()
    solver = ndist.DistPCG(device, 0, 1)
    try:
        bounds = ndist.partition_rows(table.n, 1)
        indptr, indices, data, rhs_l = solver.assemble_local(table, bounds)
        x, info = solver.solve_amg(table.n, bounds, indptr, indices, data, rhs_l, rtol=1e-10,
                                   gather_below=DIST_GATHER_BELOW)
    finally:
        solver.close()
    return x.cpu().numpy(), info


def main():
    from nodal_b200.device import Device
    device = Device.get(0)
    out = {"apply": {name: digest(apply_bits(device, name)) for name in APPLY_CASES}}
    x, info = dist_bits(device)
    out["dist_single_rank"] = {"grid": DIST_GRID, "gather_below": DIST_GATHER_BELOW, "x": digest(x),
                               "iterations": int(info["iterations"]),
                               "distributed_levels": int(info["distributed_levels"])}
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "amg_cycle_bits.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
