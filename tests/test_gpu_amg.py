"""GPU parity of the AMG-preconditioned CG (csrc/amg.cu) against its numpy statement
(tests/amg_mirror.py), scipy and the Jacobi-PCG path."""
import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

import amg_mirror as mirror
import nodal_b200 as n
import nodal_b200.equiv
from helpers import golden
from nodal_b200 import generators as gen
from test_amg_host import grid_matrix, random_network
from test_gpu_sparse import to_device_csr

pytestmark = pytest.mark.gpu
GRIDS = golden("grids.json")


def cases(name):
    if name.startswith("grid"):
        return grid_matrix(int(name[4:]))
    if name == "random":
        A = random_network(20000, 60000, 0)
    else:       # conductances over 4 / 10 decades: slow convergence, only the setup is compared for "wide"
        A = random_network(5000, 8000, 3, decades=2.0 if name == "random_mid" else 5.0)
    return A, np.random.default_rng(0).standard_normal(A.shape[0])


@pytest.mark.parametrize("name", ["grid40", "grid96", "random", "random_wide"])
def test_hierarchy_equals_numpy_statement(device, name):
    """Aggregates, coarse patterns and coarse values bit for bit on every level."""
    A, _ = cases(name)
    ref = mirror.AMG(A)
    amg = device.amg(to_device_csr(device, A))
    try:
        assert amg.rows == ref.rows
        assert amg.nnz == ref.nnz
        assert amg.direct
        for l, (Al, _, _, agg) in enumerate(ref.levels):
            assert np.array_equal(amg.aggregates(l).cpu().numpy(), agg)
        for l, Al in enumerate([lv[0] for lv in ref.levels] + [ref.Ac]):
            got = amg.operator(l).tocsr()
            Al = sps.csr_matrix(Al)
            Al.sort_indices()
            assert np.array_equal(got.indptr, Al.indptr)
            assert np.array_equal(got.indices, Al.indices)
            assert np.array_equal(got.data, Al.data)
    finally:
        amg.close()


@pytest.mark.parametrize("name", ["grid40", "grid96", "random"])
def test_cycle_equals_numpy_statement(device, name):
    A, _ = cases(name)
    r = np.random.default_rng(5).standard_normal(A.shape[0])
    want = mirror.AMG(A).cycle(r)
    amg = device.amg(to_device_csr(device, A))
    try:
        z = amg.apply(device.to_device(r)).cpu().numpy()
        z2 = amg.apply(device.to_device(r)).cpu().numpy()
    finally:
        amg.close()
    assert np.linalg.norm(z - want) <= 1e-11 * np.linalg.norm(want)
    assert np.array_equal(z, z2)                        # deterministic


@pytest.mark.parametrize("name", ["grid40", "grid96", "grid200", "random", "random_mid"])
def test_amg_pcg_solves_like_scipy(device, name):
    A, b = cases(name)
    M = mirror.AMG(A)
    _, it_ref = mirror.pcg(A, b, M)
    if name.startswith("grid"):
        x_ref = spla.spsolve(sps.csc_matrix(A), b)
    else:               # SuperLU fills in catastrophically on the random graphs: tight CG on the CPU instead
        x_ref, _ = mirror.pcg(A, b, M, rtol=1e-13)
    x, info = device.amg_pcg(to_device_csr(device, A), device.to_device(b), rtol=1e-10)
    x = x.cpu().numpy()
    assert info["status"] == 0
    assert abs(info["iterations"] - it_ref) <= max(2, it_ref // 20)
    assert info["relres"] <= 1e-10
    assert np.linalg.norm(b - A @ x) <= 1.5e-10 * np.linalg.norm(b)
    assert np.linalg.norm(x - x_ref) <= 1e-7 * np.linalg.norm(x_ref)
    assert info["levels"] == len(info["level_rows"]) >= 2
    assert info["operator_complexity"] < (1.5 if name.startswith("grid") else 3.0)


def test_small_system_is_solved_by_the_explicit_inverse(device):
    A, b = grid_matrix(12)                  # 143 unknowns <= 512: a single level
    x, info = device.amg_pcg(to_device_csr(device, A), device.to_device(b))
    assert info["levels"] == 1 and info["coarsest_direct"]
    assert info["iterations"] <= 2 and info["status"] == 0
    assert np.linalg.norm(b - A @ x.cpu().numpy()) <= 1e-10 * np.linalg.norm(b)


def test_parameters_and_edge_cases(device):
    A, b = grid_matrix(60)
    csr = to_device_csr(device, A)
    bd = device.to_device(b)
    # zero right-hand side
    x, info = device.amg_pcg(csr, device.to_device(np.zeros_like(b)))
    assert info["status"] == 0 and info["iterations"] == 0 and not x.cpu().numpy().any()
    # warm start from the solution: no iterations
    x0, _ = device.amg_pcg(csr, bd, rtol=1e-12)
    x1, info = device.amg_pcg(csr, bd, rtol=1e-10, x0=x0)
    assert info["iterations"] == 0 and np.array_equal(x0.cpu().numpy(), x1.cpu().numpy())
    # one pass per level -> pairs only, more levels; Jacobi on the coarsest level
    _, info1 = device.amg_pcg(csr, bd, passes=1, direct_max=1, coarse=64)
    ref = mirror.AMG(A, passes=1, direct_max=1, coarse=64)
    assert info1["level_rows"] == ref.rows and not info1["coarsest_direct"]
    assert info1["status"] == 0 and abs(info1["iterations"] - mirror.pcg(A, b, ref)[1]) <= 3
    # maxit
    _, info2 = device.amg_pcg(csr, bd, maxit=3)
    assert info2["status"] == 2 and info2["iterations"] == 3
    with pytest.raises(TypeError):
        device.amg(csr, nonsense=1)


def test_indefinite_matrix_is_reported(device):
    A = sps.csr_matrix(np.array([[1.0, 2.0, 0.0], [2.0, 1.0, 0.0], [0.0, 0.0, 1.0]]))
    with pytest.raises(n._lib.NodalLibraryError, match="positive definite"):
        device.amg(to_device_csr(device, A))


@pytest.mark.parametrize("key", ["grid2d_50", "grid2d_100", "lattice3d_6"])
def test_equivalent_resistance_with_amg(device, key):
    """Same R as the reference (golden) and as the Jacobi path through the public API."""
    g = GRIDS[key]
    net = gen.grid2d(g["N"]) if key.startswith("grid") else gen.lattice3d(g["N"])
    r = n.equiv.equivalent_resistance(net, "1", "g", sparse=True, precond="amg")
    assert n.equiv.equivalent_resistance.last_stats["solver"] == "amg_pcg"
    assert r == pytest.approx(g["R_sparse"], rel=1e-9)
    rj = n.equiv.equivalent_resistance(net, "1", "g", sparse=True)
    assert r == pytest.approx(rj, rel=1e-9)


def test_million_unknown_grid(device):
    """1024 x 1024: iteration count stays flat (numpy statement: 45), result equals Jacobi-PCG."""
    net = gen.grid2d(1024)
    r = n.equiv.equivalent_resistance(net, "1", "g", sparse=True, precond="amg")
    st = dict(n.equiv.equivalent_resistance.last_stats)
    assert st["status"] == 0 and st["iterations"] <= 60 and st["relres"] <= 1e-10
    rj = n.equiv.equivalent_resistance(net, "1", "g", sparse=True)
    assert r == pytest.approx(rj, rel=1e-9)


@pytest.mark.parametrize("mode", ["dense", "jacobi", "amg"])
def test_many_port_equivalent_resistances(device, mode):
    """SURVEY 8(f) rank 4: one assembly (and one AMG hierarchy), many (a, b) pairs; every value
    equals the single-pair call of the reference API and the oracle."""
    from oracle import mna_oracle as orc
    N = 30
    net = gen.grid2d(N)
    pairs = [("1", "g"), ("g", "1"), ("n0_0", "n29_29"), ("n3_4", "1"), ("n7_7", "n7_7"), ("n10_2", "g")]
    kw = dict(sparse=False) if mode == "dense" else dict(sparse=True, precond=mode, rtol=1e-12)
    if mode == "amg":
        kw["amg"] = dict(coarse=64)                     # 899 unknowns: force a real hierarchy
    got = n.equiv.equivalent_resistances(net, pairs, **kw)
    stats = n.equiv.equivalent_resistances.last_stats
    assert len(got) == len(stats) == len(pairs)
    rows = orc.grid2d_rows(N)
    for (a, b), r, st in zip(pairs, got, stats):
        if a == b:
            assert r == 0.0
            continue
        want = orc.equivalent_resistance(rows, a, b, sparse=True)
        assert r == pytest.approx(want, rel=1e-9)
        assert r == pytest.approx(n.equiv.equivalent_resistance(net, a, b, **kw), rel=1e-9)
        if mode == "amg":       # several pairs: the batched solver (all right-hand sides advance together)
            assert st["solver"] == "amg_pcg_multi" and len(st["level_rows"]) >= 2 and st["relres"] <= 1e-12
    assert got[0] == pytest.approx(got[1], rel=1e-12)    # symmetric in (a, b)
    with pytest.raises(KeyError):
        n.equiv.equivalent_resistances(net, [("1", "nowhere")], **kw)


# ------------------------------------------------------------------ row-partitioned form, one rank
@pytest.mark.parametrize("N,amg", [(100, {}), (100, {"gather_below": 400}), (100, {"gather_below": 3000, "passes": 1}),
                                   (400, {"gather_below": 5000}), (1000, {"gather_below": 20000}),
                                   ("random", {"gather_below": 2000})])
def test_dist_amg_single_rank(device, N, amg):
    """csrc/dist_amg.cu with a world of one rank (empty halos, no exchange) must reproduce the
    single-GPU hierarchy: same level sizes where the levels are built the same way, same answer.
    The random network's distributed levels are too dense for the member-row merge (amg_merge_pays
    is false): their products go through the sort-based builder."""
    import copy
    from nodal_b200 import dist as ndist
    net = copy.deepcopy(gen.random_network(20000, degree=8, seed=1) if N == "random" else gen.grid2d(N))
    net.process_component(["a1", "A", "1", "1", "g"])
    table = net.table()
    csr, rhs = device.assemble_csr(table)
    x1, i1 = device.amg_pcg(csr, rhs, rtol=1e-10, **{k: v for k, v in amg.items() if k != "gather_below"})
    solver = ndist.DistPCG(device, 0, 1)
    try:
        bounds = ndist.partition_rows(table.n, 1)
        indptr, indices, data, rhs_l = solver.assemble_local(table, bounds)
        x, info = solver.solve_amg(table.n, bounds, indptr, indices, data, rhs_l, rtol=1e-10, **amg)
    finally:
        solver.close()
    assert info["status"] == 0 and info["relres"] <= 1e-10, info
    if "gather_below" in amg:
        assert info["distributed_levels"] >= 1, info
    # one rank: the aggregates are the single-GPU ones, level for level
    # (the distributed coarsening stops at gather_below, the single-GPU one at `coarse` rows)
    common = min(len(info["level_rows"]), len(i1["level_rows"]))
    assert info["level_rows"][:common] == i1["level_rows"][:common], (info, i1)
    assert abs(info["iterations"] - i1["iterations"]) <= 4
    if N == "random":       # no pinned value: the single-GPU solve is the reference
        assert float((x - x1).abs().max()) <= 1e-9 * float(x1.abs().max())
    else:
        want = {100: GRIDS["grid2d_100"]["R_sparse"], 400: 0.7732566450916762, 1000: 0.7732422803670024}[N]
        assert float(x[net.nodenum["1"]]) == pytest.approx(want, rel=1e-9)
    resid = device.spmv(csr, x) - rhs
    assert float(resid.norm() / rhs.norm()) <= 1.05e-10
    assert float((x - x1).abs().max()) <= 1e-8 * float(x1.abs().max())


def test_multi_rhs_solver_matches_single_solves(device):
    """csrc/amg_multi.cu: K right-hand sides against one hierarchy, each equal to its own single
    solve (to the tolerance) with a similar iteration count; zero and duplicate right-hand sides,
    more than one batch, and the single-pair path of port_resistances stay consistent."""
    import torch
    net = gen.grid2d(120)
    table = net.table()
    csr, _ = device.assemble_csr(table)
    amg = device.amg(csr)
    try:
        rng = np.random.default_rng(5)
        K = 8
        rhs = torch.zeros(K, csr.n, dtype=torch.float64, device="cuda")
        picks = rng.choice(csr.n, size=(K, 2), replace=False)
        for k in range(K):
            rhs[k, picks[k, 0]] = 1.0
            rhs[k, picks[k, 1]] = -1.0
        rhs[3] = 0.0                                   # b = 0 -> x = 0, no iterations
        rhs[5] = rhs[1]                                # duplicates converge together
        xs, infos = amg.solve_multi(rhs, rtol=1e-11)
        for k in range(K):
            assert infos[k]["status"] == 0 and infos[k]["relres"] <= 1e-11, infos[k]
            if k == 3:
                assert infos[k]["iterations"] == 0 and float(xs[k].abs().max()) == 0.0
                continue
            x1, i1 = amg.solve(rhs[k].clone(), rtol=1e-11)
            assert abs(infos[k]["iterations"] - i1["iterations"]) <= 3
            assert float((xs[k] - x1).abs().max()) <= 1e-8 * float(x1.abs().max())
            resid = device.spmv(csr, xs[k].contiguous()) - rhs[k]
            assert float(resid.norm() / rhs[k].norm()) <= 1.05e-11
        assert torch.equal(xs[5], xs[1])
    finally:
        amg.close()
    # 11 pairs = two batches; equal to pair-by-pair solves
    pairs = [("1", "g")] + [(f"n{3 * k}_{2 * k}", f"n{100 - k}_{90 - 2 * k}") for k in range(10)]
    batched = n.equiv.equivalent_resistances(net, pairs, sparse=True, precond="amg")
    assert all(st["solver"] == "amg_pcg_multi" for st in n.equiv.equivalent_resistances.last_stats)
    single = n.equiv.equivalent_resistances(net, pairs, sparse=True, precond="amg", multi_rhs=False)
    assert all(st["solver"] == "amg_pcg" for st in n.equiv.equivalent_resistances.last_stats)
    for rb, rs in zip(batched, single):
        assert rb == pytest.approx(rs, rel=1e-8)
