"""Row-partitioned eliminated solve (nodal_b200/dist_sources.py), checked on every rank (not a pytest
file; tests/test_gpu_dist_sources.py runs it under torchrun on 1 and 2 GPUs):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29541 tests/dist_sources_check.py

1. the rank's rows of the full MNA matrix, the replicated forest and the rank's reduced rows are
   bit-identical to the single-GPU assemble_csr, source_forest and source_reduce + assemble_csr_raw;
2. the staged expansion of the single-GPU reduced solution gives x byte-equal to source_expand, and
   relres_full to 1e-12;
3. Circuit(net, sparse=True, distributed=True, rtol=1e-12).solve() on the CASES netlists and on
   power_grid(200, 16) against the oracle, and bitwise equal on a second run;
4. power_grid(2048, 64) (2 ranks and more): source currents against the load, potentials <= vdd, and
   ||A - G x|| from the ranks' rows;
5. a loop of sources, eliminate_sources=False and a VCVS netlist raise NotImplementedError;
6. the R / A path: assemble_from_host gives the single-GPU rows of grid2d(100)."""
import copy
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import nodal_b200 as n  # noqa: E402
from helpers import block_err, write_csv  # noqa: E402
from nodal_b200 import constants as K  # noqa: E402
from nodal_b200 import dist as ndist  # noqa: E402
from nodal_b200 import generators as gen  # noqa: E402
from nodal_b200.device import Device, DeviceCSR  # noqa: E402
from oracle import mna_oracle as orc  # noqa: E402
from test_sources_host import CASES, case_rows  # noqa: E402

RANK = WORLD = 0
OK = True


def report(**msg):
    global OK
    OK &= bool(msg.get("ok", True))
    if RANK == 0 or not msg.get("ok", True):
        print(json.dumps(dict(rank=RANK, world=WORLD, **msg)), flush=True)


def rows_of(net):
    t = net.table()
    nodes = list(net.nodenum) + [net.ground]
    keys = net.component_keys
    return [[keys[k], K.TYPE_NAME[int(t.type[k])], repr(float(t.value[k])), nodes[t.a[k]], nodes[t.b[k]]]
            for k in range(len(t))]


def same(a, b):
    return a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()


def rows_equal(local, rhs_local, csr, rhs, bounds):
    """LocalRows + rhs slice against rows [rb, re) of a whole CSR, byte for byte."""
    rb, re = int(bounds[RANK]), int(bounds[RANK + 1])
    ip = csr.indptr[rb: re + 1]
    s, e = int(ip[0]), int(ip[-1])
    return (same(local.indptr, ip - ip[0]) and same(local.indices, csr.indices[s:e]) and same(local.data, csr.data[s:e])
            and same(rhs_local, rhs[rb:re]))


def broadcast(t):
    if WORLD > 1:
        dist.broadcast(t, src=0)
    return t


def check_parts(name, net, dev):
    """Checks 1 and 2 against this rank's own single-GPU computation."""
    table = net.table()
    kcl = table.kcl
    dtab = dev.upload_table(table)
    csr, rhs = dev.assemble_csr(table, dtab=dtab)
    finfo, f = dev.source_forest(dtab, len(table), kcl, table.be)
    red, nred = dev.source_reduce(dtab, len(table), kcl, f)
    m = finfo["rows"]
    rcsr, rrhs = dev.assemble_csr_raw(red, nred, m, m, 4)

    circuit = n.Circuit(net, sparse=True, distributed=True, rtol=1e-12)
    d = circuit._dsrc
    full_ok = rows_equal(circuit.G, circuit.A, csr, rhs, d.bounds)
    info2, f2, etab = d.forest()
    forest_ok = info2 == finfo
    for k in ("rep_row", "offset", "depth"):
        forest_ok &= same(f2[k], f[k])
    forest_ok &= same(f2["roots"][:m], f["roots"][:m])
    # parent_edge indexes the E-only table there: mapped through the E rows' table rows it is the whole table's
    erow = f["erow"][: finfo["sources"]].long()
    pe = f2["parent_edge"].long()
    mapped = torch.where(pe >= 0, erow[pe.clamp(min=0)] if len(erow) else pe, pe).int()
    forest_ok &= same(mapped, f["parent_edge"])
    stats = {}
    rows, rrhs_local = d.reduced_rows(f2, m, stats)
    reduced_ok = stats["reduced_components"] == nred and rows_equal(rows, rrhs_local, rcsr, rrhs,
                                                                    ndist.partition_rows(m, WORLD))
    # staged expansion of one reduced solution (rank 0's) against the single-GPU expansion of it
    y, _ = dev.pcg(rcsr, rrhs, rtol=1e-12)
    y = broadcast(y.contiguous())
    x1, relres1 = dev.source_expand(dtab, kcl, f, finfo, y, csr, rhs)
    x2 = d.expand(info2, f2, etab, y)
    relres2 = d.relres(x2)
    expand_ok = same(x1, x2) and abs(relres2 - relres1) <= 1e-12 * max(relres1, 1e-300)
    report(check="rows, forest, reduced rows, staged expansion", net=name, full_rows=full_ok, forest=forest_ok,
           reduced_rows=reduced_ok, expansion_bytes=expand_ok, relres_single=relres1, relres_staged=relres2,
           ok=full_ok and forest_ok and reduced_ok and expand_ok)


def check_solve(name, net, rows):
    """Check 3: the public surface against the oracle, and a bitwise rerun."""
    _, _, _, _, want = orc.solve_rows(rows, sparse=True, backend="dict")
    kcl = net.nums["kcl"]
    a = n.Circuit(net, sparse=True, distributed=True, rtol=1e-12).solve()
    b = n.Circuit(net, sparse=True, distributed=True, rtol=1e-12).solve()
    red = a.stats["reduction"]
    err_e = block_err(a.result[:kcl], want[:kcl], kcl)
    err_i = block_err(a.result[kcl:], want[kcl:], 0)
    good = (red["eliminated"] and a.stats["status"] == 0 and red["relres_full"] <= 1e-9 and red["world"] == WORLD
            and len(a.result) == net.table().n and err_e <= 1e-9 and err_i <= 1e-9
            and a.result.tobytes() == b.result.tobytes())
    report(check="Circuit(distributed=True).solve() vs oracle", net=name, solver=a.stats["solver"],
           iterations=a.stats["iterations"], relres_full=red["relres_full"], err_potentials=err_e, err_currents=err_i,
           rerun_bitwise=a.result.tobytes() == b.result.tobytes(), ok=good)


def check_large(dev):
    """Check 4 on power_grid(2048, 64)."""
    vdd = 1.0
    net = gen.power_grid(2048, 64, vdd=vdd, load=1e-4, seed=0)
    table = net.table()
    circuit = n.Circuit(net, sparse=True, distributed=True, rtol=1e-12)
    sol = circuit.solve()
    x = sol.result
    load = float(table.value[table.type == K.T_A].sum())
    cur = abs(float(x[table.kcl:].sum()) - load) / load
    G = circuit.G
    gx = dev.spmv(DeviceCSR(G.shape[0], G.indptr, G.indices, G.data), dev.to_device(x))
    sums = torch.stack([((circuit.A - gx) ** 2).sum(), (circuit.A ** 2).sum()])
    if WORLD > 1:
        dist.all_reduce(sums)
    rel = float(torch.sqrt(sums[0] / sums[1]))
    red = sol.stats["reduction"]
    good = sol.stats["status"] == 0 and cur <= 1e-9 and bool(np.all(x[: table.kcl] <= vdd)) and rel <= 1e-9
    report(check="power_grid(2048, 64)", unknowns=table.n, current_vs_load=cur, relres_local_rows=rel,
           relres_full=red["relres_full"], iterations=sol.stats["iterations"],
           split_ms={k: red[k] for k in ("upload_ms", "full_assemble_ms", "forest_ms", "reduce_ms", "assemble_ms",
                                          "solve_ms", "expand_ms", "relres_ms")}, ok=good)


def check_refusals(tmp):
    def raises(rows, fname, **opts):
        net = n.Netlist(write_csv(rows, os.path.join(tmp, fname)))
        try:
            n.Circuit(net, sparse=True, distributed=True, **opts).solve()
        except NotImplementedError as err:
            return str(err)
        return None
    loop = raises(case_rows("pads") + [["vp", "E", "1.0", "n0_0", "g"]], "loop.csv")
    off = raises(case_rows("pads"), "off.csv", eliminate_sources=False)
    vcvs = raises(orc.grid2d_rows(8) + [["v1", "E", "1", "n0_0", "g"], ["d1", "VCVS", "2", "n5_5", "g", "n0_0", "g"]],
                  "vcvs.csv")
    good = loop is not None and "forest" in loop and off is not None and vcvs is not None
    report(check="NotImplementedError", loop=loop, eliminate_sources_false=off, vcvs=vcvs, ok=good)


def check_ra_path(dev):
    net = copy.deepcopy(gen.grid2d(100))
    net.process_component(["a1", "A", "1", "1", "g"])
    table = net.table()
    runner = ndist.GridRunner(dev, table, net.nodenum["1"], RANK, WORLD, solver=ndist.shared_solver(dev, RANK, WORLD))
    a = runner.assemble(dev.upload_table(table))
    b = runner.assemble_from_host()
    csr, rhs = dev.assemble_csr(table)
    local = ndist.LocalRows(table.n, runner.bounds, RANK, *b[:3])
    good = all(torch.equal(u, v) for u, v in zip(a, b)) and rows_equal(local, b[3], csr, rhs, runner.bounds)
    report(check="R / A assemble_from_host == single-GPU rows", N=100, ok=good)


def main():
    global RANK, WORLD
    RANK, WORLD, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = Device.get(local)
    with tempfile.TemporaryDirectory() as tmp:
        tmp = os.path.join(tmp, f"rank{RANK}")
        os.makedirs(tmp)
        for case in CASES:
            rows = case_rows(case)
            net = n.Netlist(write_csv(rows, os.path.join(tmp, f"{case}.csv")))
            check_parts(case, net, dev)
            check_solve(case, net, rows)
        pg = gen.power_grid(200, 16, vdd=1.0, load=1e-3, seed=1)
        check_parts("power_grid(200, 16)", pg, dev)
        check_solve("power_grid(200, 16)", pg, rows_of(pg))
        if WORLD >= 2:
            check_large(dev)
        check_refusals(tmp)
        check_ra_path(dev)
    flag = torch.tensor([1 if OK else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if RANK == 0:
        print("DIST_SOURCES_CHECK", "PASS" if flag.item() else "FAIL", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
