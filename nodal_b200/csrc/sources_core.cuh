// Per-item rules of the independent-voltage-source elimination (csrc/sources.cu), written once as
// __host__ __device__ functions so the GPU kernels and the CPU-side check
// (tests/host_check/sources_host.cpp against tests/sources_mirror.py) share them.
//
// Every E row fixes e_a - e_b = V.  When the E rows form a forest over the nodes (ground is node
// kcl), every node of a tree has the potential y_root + offset; a tree holding ground has y_root = 0.
// The R / A rows then reduce to an R / A table over the roots (a weighted graph Laplacian, SPD),
// and the source currents come back from KCL summed over the subtree each source cuts off.
#pragma once
#include <stdint.h>

#include "schur_core.cuh"

#ifndef __CUDACC__
#define __host__
#define __device__
#endif

// lead index of the component table -> node of the source forest (ground is node kcl)
__host__ __device__ inline int32_t src_node(int32_t lead, int32_t kcl) { return lead < 0 ? kcl : lead; }

// offset of a child across a source of value v: e_a - e_b = v
__host__ __device__ inline double src_child_offset(double parent_offset, double v, bool child_is_anode) {
    return child_is_anode ? parent_offset + v : parent_offset - v;
}

// Rows the reduced table gets for one component (at most two, in this order):
//   R(a, b)   -> R(A, B) and, if the offsets of a and b differ, A(-(o_a - o_b) / R) between A and B
//                (the current the fixed offsets drive through the resistor); nothing if A == B
//   A(a, b)   -> A(A, B); nothing if A == B
//   any other -> nothing (E rows are what is eliminated)
// A, B = rep_row[node]: the reduced row of the lead's tree, or -1 (GROUND) for the tree of ground.
struct ReducedRows {
    uint8_t type[2];
    double value[2];
    int32_t a[2], b[2];
    int count;
};

__host__ __device__ inline void src_reduce_component(int type, double value, int32_t a, int32_t b, int32_t kcl,
                                                     const int32_t* rep_row, const double* offset,
                                                     ReducedRows& o) {
    o.count = 0;
    if (type != 0 && type != 1) return;
    const int32_t na = src_node(a, kcl), nb = src_node(b, kcl);
    const int32_t ra = rep_row[na], rb = rep_row[nb];
    if (ra == rb) return;
    o.type[0] = (uint8_t)type; o.value[0] = value; o.a[0] = ra; o.b[0] = rb; o.count = 1;
    if (type == 0) {
        const double oa = offset[na], ob = offset[nb];
        if (oa != ob) {
            o.type[1] = 1; o.value[1] = -(oa - ob) / value; o.a[1] = ra; o.b[1] = rb; o.count = 2;
        }
    }
}

__host__ __device__ inline int src_reduce_count(int type, int32_t a, int32_t b, int32_t kcl,
                                                const int32_t* rep_row, const double* offset) {
    if (type != 0 && type != 1) return 0;
    const int32_t na = src_node(a, kcl), nb = src_node(b, kcl);
    if (rep_row[na] == rep_row[nb]) return 0;
    return (type == 0 && offset[na] != offset[nb]) ? 2 : 1;
}

// potential of a node from the reduced solution y
__host__ __device__ inline double src_potential(int32_t rep, double offset, const double* y) {
    return (rep < 0 ? 0.0 : y[rep]) + offset;
}

// current of the source between a child and its parent from the KCL residual summed over the
// child's subtree (the reference's sign: the branch current enters the anode's KCL row with -1)
__host__ __device__ inline double src_current(double subtree_sum, bool child_is_anode) {
    return child_is_anode ? -subtree_sum : subtree_sum;
}

// ---------------------------------------------------------------- E rows plus dependent branch rows
// (nodal_b200/source_schur.py; tests/source_schur_mirror.py states it in numpy)
//
// With dependent sources (VCVS, VCCS, CCVS, CCCS, the VCVS of an OPMODEL) the forest is built on the
// E rows alone and the reduced system gets one more unknown per dependent branch: m_n node rows (the
// reduced rows above) then m_d dependent branch rows, numbered in branch order by d_map (branch ->
// dependent index, -1 for the E branches).  Its node-node block and node right-hand side are the stamp
// of the reduced R / A table; every other entry comes from one row of the full sorted MNA matrix G,
// in CSR order, as mapped below.  The reference resolves collisions inside a branch row by
// overwriting, so the mapped leads are not re-stamped: the entries of the full rows are summed per
// reduced column by the CSR build, in emission order.
//   node row i outside ground's tree:  G[i, kcl + k] with d_map[k] >= 0  ->  (rep_row[i], m_n + d_map[k])
//                                      (node and E columns: the reduced table's part / cancelled)
//   dependent branch row kcl + k:      G[., j], j a node  ->  (m_n + d, rep_row[j]), dropped in ground's tree
//                                      G[., kcl + k'], d_map[k'] >= 0  ->  (m_n + d, m_n + d_map[k'])
//                                      and the right-hand side (m_n + d, nr): A - sum_j G[., j] o_j over
//                                      the node columns (schur_branch_rhs with the offsets)
//   every other row (ground's tree, E branch rows): nothing
// Stamping never puts an E column into a dependent branch row.

template <class Sink>
__host__ __device__ inline void src_dep_row(int32_t i, const int32_t* indptr, const int32_t* indices,
                                            const double* data, const double* rhs, int32_t kcl,
                                            const int32_t* rep_row, const double* offset, const int32_t* d_map,
                                            int32_t mn, int32_t nr, Sink& out) {
    const int64_t begin = indptr[i], end = indptr[i + 1];
    if (i < kcl) {
        const int32_t r = rep_row[i];
        if (r < 0) return;
        for (int64_t p = begin; p < end; ++p) {
            const int32_t c = indices[p];
            if (c >= kcl && d_map[c - kcl] >= 0) out(r, mn + d_map[c - kcl], data[p]);
        }
        return;
    }
    const int32_t d = d_map[i - kcl];
    if (d < 0) return;
    for (int64_t p = begin; p < end; ++p) {
        const int32_t c = indices[p];
        if (c < kcl) {
            if (rep_row[c] >= 0) out(mn + d, rep_row[c], data[p]);
        } else if (d_map[c - kcl] >= 0) {
            out(mn + d, mn + d_map[c - kcl], data[p]);
        }
    }
    out(mn + d, nr, schur_branch_rhs(indices, data, begin, end, kcl, rhs[i], offset));
}

// a VCVS / VCCS / CCVS whose two output leads lie in one source tree: its branch row loses its
// incidence and its current is undetermined (the full system is singular too)
__host__ __device__ inline bool src_dep_collapsed(int type, int32_t a, int32_t b, int32_t kcl, const int32_t* rep_row) {
    if (type != 3 && type != 4 && type != 5) return false;
    return rep_row[src_node(a, kcl)] == rep_row[src_node(b, kcl)];
}
