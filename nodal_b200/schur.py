"""Sparse solve of netlists with op-amps and dependent sources through the Schur complement of the
branch rows.

In MNA form G = [[L, B], [C, D]]: the first kcl rows and columns are the node rows, the last m the
branch rows, and only resistors stamp into the node-node block, so L is the resistor Laplacian (SPD
when every node reaches ground through resistors).  Block elimination is exact: with
S = D - C L^-1 B (m x m), one application of the block inverse to (r_n, r_b) is

    t = L^-1 r_n,   x_b = S^-1 (r_b - C t),   x_n = L^-1 (r_n - B x_b).

L^-1 B costs ceil(m / 8) batched AMG solves (csrc/amg_multi.cu), S goes through the dense LU once
(csrc/lu_dense.cu), and iterative refinement on the full system, x += M^-1 (A - G x) from x = 0,
recovers the accuracy that cond(S) costs (op-amp gains make S badly conditioned).  The split, the
columns of S and the couplings run in csrc/schur.cu; tests/schur_mirror.py states the algorithm in
numpy.  Without it such netlists go to GMRES with a diagonal preconditioner, which stalls on the
branch rows: above the dense-LU limit that ends in NaNs.

Circuit(netlist, sparse=True, schur=...):
    False  (default) the existing path
    True   solve through the Schur complement when the netlist qualifies: at least one branch row,
           every R positive, every node reaching ground through resistors alone and
           m <= schur_max_branches (default 8192; S and its factors are m^2 doubles).  Otherwise,
           or when the refinement does not reach rtol, the existing path runs and
           Solution.stats["schur"]["reason"] says why.
    schur_rtol (default rtol) is the tolerance of the L solves, schur_refine (default 5) the most
    applications of the block inverse.  A step that does not halve the residual ends the refinement.
"""
from __future__ import annotations

import math
import time

from . import _lib


def check_option(options, sparse, distributed):
    """Validate schur and its parameters; True with sparse=False or distributed=True is an error."""
    mode = options.get("schur", False)
    if mode is not True and mode is not False:
        raise ValueError(f"schur must be True or False, got {mode!r}")
    if mode and not sparse:
        raise ValueError("schur=True needs sparse=True (the dense path already solves by LU)")
    if mode and distributed:
        raise NotImplementedError("the Schur-complement solve runs on one GPU (distributed=True is not supported)")
    if int(options.get("schur_refine", 5)) < 0:
        raise ValueError("schur_refine must be >= 0")
    if int(options.get("schur_max_branches", 8192)) < 1:
        raise ValueError("schur_max_branches must be >= 1")
    return mode


def skip_reason(table, max_branches):
    """"" when the table qualifies as far as the host can tell, else why not (the connectivity of the
    resistors is decided on the device, in solve())."""
    if table.be == 0:
        return "no branch rows"
    f = table.facts()
    if f["unknown_type"]:
        return "unknown component type"
    if f["r_nonpositive"]:
        return "a resistance is not positive (L would not be SPD)"
    if table.be > max_branches:
        return f"{table.be} branch rows > schur_max_branches ({max_branches})"
    return ""


def _ms(t0, dev):
    dev.torch.cuda.current_stream(dev.dev).synchronize()
    return (time.perf_counter() - t0) * 1e3


def solve(circuit):
    """(x, info) of the full system through the Schur complement, or (None, stats) when it is not
    requested (stats None), does not apply or does not converge (stats["reason"] says why)."""
    if not circuit._schur:
        return None, None
    table, dev, opts = circuit.table, circuit._dev, circuit.options
    kcl, m = table.kcl, table.be
    stats = dict(applied=False, branches=m, node_rows=kcl)
    reason = skip_reason(table, int(opts.get("schur_max_branches", 8192)))
    if reason:
        stats["reason"] = reason
        return None, stats
    if getattr(circuit, "_G_sorted", None) is not None:     # as in Circuit._device_solve
        circuit.G, circuit._G_sorted = circuit._G_sorted, None
    G, A = circuit.G, circuit.A
    rtol = opts.get("rtol", 1e-10)
    inner = opts.get("schur_rtol", rtol)
    refine = int(opts.get("schur_refine", 5))
    maxit = opts.get("maxit")

    t0 = time.perf_counter()
    grounded = dev.r_grounded(circuit._dtab, len(table), kcl)
    stats["check_ms"] = _ms(t0, dev)
    if not grounded:
        stats["reason"] = "a node does not reach ground through resistors (L would be singular)"
        return None, stats
    t0 = time.perf_counter()
    L, B = dev.schur_split(G, kcl)
    stats["split_ms"] = _ms(t0, dev)
    t0 = time.perf_counter()
    try:
        amg = dev.amg(L, **(opts.get("amg") or {}))
    except _lib.NodalLibraryError as err:
        stats["reason"] = f"AMG setup on L failed: {err}"
        return None, stats
    stats["amg_setup_ms"] = _ms(t0, dev)
    try:
        return _solve_with(dev, amg, G, A, B, kcl, m, rtol, inner, refine, maxit, stats)
    finally:
        amg.close()


def _solve_with(dev, amg, G, A, B, kcl, m, rtol, inner, refine, maxit, stats):
    torch = dev.torch
    # ---- columns of S, eight at a time
    t0 = time.perf_counter()
    S = dev.empty(m * m, torch.float64).view(m, m)
    batches, worst = 0, 0
    for j0 in range(0, m, 8):
        K = min(8, m - j0)
        Z, infos = amg.solve_multi(dev.schur_rhs_batch(kcl, j0, K, B), rtol=inner, maxit=maxit)
        batches += 1
        worst = max([worst] + [i["iterations"] for i in infos])
        bad = [i for i in infos if i["status"] != 0]
        if bad:
            stats.update(batches=batches, batch_iterations_max=worst)
            stats["reason"] = (f"the L solves of branch columns {j0}..{j0 + K - 1} did not converge "
                               f"(status {bad[0]['status']}, relres {bad[0]['relres']:.1e})")
            return None, stats
        dev.schur_columns(G, kcl, j0, Z, S)
        del Z
    stats.update(batches=batches, batch_iterations_max=worst, columns_ms=_ms(t0, dev))
    # ---- S = P^T L U once
    t0 = time.perf_counter()
    ipiv, finfo = dev.lu_factor(S)
    stats["factor_ms"] = _ms(t0, dev)
    if finfo["status"] != 0:
        stats["reason"] = f"S is singular (zero pivot {finfo['info']})"
        return None, stats
    # ---- refinement from x = 0
    n = kcl + m
    x = dev.zeros(max(2, n), torch.float64)[:n]
    r = dev.empty(max(2, n), torch.float64)[:n]
    history, step_ms, inner_its = [], [], 0
    reason = ""
    step = 0
    while True:
        rr, bb = dev.schur_residual(G, A, x, r)
        relres = math.sqrt(rr / bb) if bb > 0 else (0.0 if rr == 0 else math.inf)
        history.append(relres)
        if relres <= rtol:
            break
        if step == refine:
            reason = f"relres {relres:.2e} > rtol {rtol:.1e} after {refine} refinement step(s)"
            break
        if step >= 1 and not relres <= 0.5 * history[-2]:
            reason = f"refinement step {step} did not halve the residual ({history[-2]:.2e} -> {relres:.2e})"
            break
        t0 = time.perf_counter()
        t, it1 = amg.solve(r[:kcl], rtol=inner, maxit=maxit)
        xb = dev.lu_solve_factored(S, ipiv, dev.schur_branch_rhs(G, kcl, r, t))
        xn, it2 = amg.solve(dev.schur_node_rhs(kcl, B, r, xb), rtol=inner, maxit=maxit)
        if it1["status"] != 0 or it2["status"] != 0:
            reason = f"an L solve of refinement step {step + 1} did not converge"
            break
        inner_its += it1["iterations"] + it2["iterations"]
        dev.schur_add(x[:kcl], xn)
        dev.schur_add(x[kcl:], xb)
        step += 1
        step_ms.append(_ms(t0, dev))
    stats.update(refine_steps=step, refine_ms=step_ms, relres_history=history, relres_full=history[-1],
                 refine_iterations=inner_its)
    if reason:
        stats["reason"] = reason
        return None, stats
    stats.update(applied=True, reason="")
    return x, dict(solver="schur", status=0, iterations=step, relres=history[-1], schur=stats)
