// TEST-ONLY: compiles the __host__ __device__ rules of the solve with E rows and dependent branch
// rows (nodal_b200/csrc/sources_core.cuh src_dep_row, src_dep_collapsed) for the CPU with contraction
// off, driven row by row as the kernels of csrc/sources.cu drive them, so that `pytest -m "not gpu"`
// checks them bit for bit against tests/source_schur_mirror.py.  Not part of the product library.
#include <stdint.h>

#include "../../nodal_b200/csrc/sources_core.cuh"

struct Count {
    int64_t n = 0;
    void operator()(int32_t, int32_t, double) { ++n; }
};

struct Store {
    int64_t* row;
    int64_t* col;
    double* val;
    int64_t p;
    void operator()(int32_t r, int32_t c, double v) {
        row[p] = r;
        col[p] = c;
        val[p] = v;
        ++p;
    }
};

// the triples of every row in row order: pass null outputs to get the count only
extern "C" int64_t source_dep_triples_host(int32_t n, int32_t kcl, const int32_t* indptr, const int32_t* indices,
                                           const double* data, const double* rhs, const int32_t* rep_row,
                                           const double* offset, const int32_t* d_map, int32_t mn, int32_t nr,
                                           int64_t* row, int64_t* col, double* val) {
    int64_t p = 0;
    for (int32_t i = 0; i < n; ++i) {
        if (!row) {
            Count c;
            src_dep_row(i, indptr, indices, data, rhs, kcl, rep_row, offset, d_map, mn, nr, c);
            p += c.n;
        } else {
            Store s{row, col, val, p};
            src_dep_row(i, indptr, indices, data, rhs, kcl, rep_row, offset, d_map, mn, nr, s);
            p = s.p;
        }
    }
    return p;
}

extern "C" int64_t source_dep_collapsed_host(int64_t ncomp, const uint8_t* type, const int32_t* a, const int32_t* b,
                                             int32_t kcl, const int32_t* rep_row) {
    int64_t c = 0;
    for (int64_t i = 0; i < ncomp; ++i) c += src_dep_collapsed(type[i], a[i], b[i], kcl, rep_row) ? 1 : 0;
    return c;
}
