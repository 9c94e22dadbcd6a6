// TEST-ONLY: compiles the __host__ __device__ rules of the voltage-source elimination
// (nodal_b200/csrc/sources_core.cuh) for the CPU, driven in the device's orders, so that
// `pytest -m "not gpu"` checks them bit for bit against tests/sources_mirror.py.  Not part of the
// product library.
#include <stdint.h>

#include "../../nodal_b200/csrc/sources_core.cuh"

// offsets from parent_edge, visiting the nodes in `order` (parents before children)
extern "C" void src_offsets_host(int32_t count, const int32_t* order, const int32_t* parent_edge, const double* value,
                                 const int32_t* a, const int32_t* b, int32_t kcl, double* offset) {
    for (int32_t k = 0; k < count; ++k) {
        const int32_t w = order[k], r = parent_edge[w];
        if (r < 0) { offset[w] = 0.0; continue; }
        const int32_t na = src_node(a[r], kcl), nb = src_node(b[r], kcl);
        const int32_t parent = na == w ? nb : na;
        offset[w] = src_child_offset(offset[parent], value[r], na == w);
    }
}

// the reduced table in component order; returns its number of rows
extern "C" int64_t src_reduce_table_host(int64_t ncomp, const uint8_t* type, const double* value, const int32_t* a,
                                         const int32_t* b, int32_t kcl, const int32_t* rep_row, const double* offset,
                                         uint8_t* o_type, double* o_value, int32_t* o_a, int32_t* o_b) {
    int64_t p = 0;
    for (int64_t i = 0; i < ncomp; ++i) {
        ReducedRows o;
        src_reduce_component(type[i], value[i], a[i], b[i], kcl, rep_row, offset, o);
        if (o.count != src_reduce_count(type[i], a[i], b[i], kcl, rep_row, offset)) return -1;
        for (int k = 0; k < o.count; ++k, ++p) {
            o_type[p] = o.type[k]; o_value[p] = o.value[k]; o_a[p] = o.a[k]; o_b[p] = o.b[k];
        }
    }
    return p;
}

// x = [e; i] from y and the KCL residual rho (kcl entries; clobbered into the subtree sums)
extern "C" void src_expand_host(int32_t kcl, int32_t n, const int32_t* rep_row, const double* offset,
                                const int32_t* parent_edge, const int32_t* depth, int32_t max_depth, const int32_t* a,
                                const int32_t* b, const int32_t* branch, const double* y, double* rho, double* x) {
    for (int32_t v = 0; v < n; ++v) x[v] = v < kcl ? src_potential(rep_row[v], offset[v], y) : 0.0;
    for (int32_t d = max_depth; d >= 1; --d)
        for (int32_t w = 0; w < kcl; ++w) {
            if (depth[w] != d) continue;
            const int32_t r = parent_edge[w];
            const int32_t na = src_node(a[r], kcl), nb = src_node(b[r], kcl);
            x[kcl + branch[r]] = src_current(rho[w], na == w);
            const int32_t parent = na == w ? nb : na;
            if (parent < kcl) rho[parent] = rho[parent] + rho[w];
        }
}
