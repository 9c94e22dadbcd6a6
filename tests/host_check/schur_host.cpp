// TEST-ONLY: compiles the __host__ __device__ rules of the Schur-complement solve
// (nodal_b200/csrc/schur_core.cuh) for the CPU with contraction off, driven row by row as the
// kernels of csrc/schur.cu drive them, so that `pytest -m "not gpu"` checks them bit for bit against
// tests/schur_mirror.py.  Not part of the product library.
#include <stdint.h>

#include "../../nodal_b200/csrc/schur_core.cuh"

// L and the B lists of the node rows (row pointers already scanned by the caller from the counts)
extern "C" void schur_counts_host(int32_t kcl, const int32_t* indptr, const int32_t* indices, int32_t* lcount,
                                  int32_t* bcount) {
    for (int32_t i = 0; i < kcl; ++i) {
        lcount[i] = schur_l_count(indices, indptr[i], indptr[i + 1], kcl);
        bcount[i] = indptr[i + 1] - indptr[i] - lcount[i];
    }
}

extern "C" void schur_columns_host(int32_t kcl, int32_t m, int32_t j0, int32_t K, const int32_t* indptr,
                                   const int32_t* indices, const double* data, const double* Z, double* S) {
    for (int32_t r = 0; r < m; ++r)
        for (int32_t k = 0; k < K; ++k)
            S[(int64_t)r * m + j0 + k] =
                schur_column_entry(indices, data, indptr[kcl + r], indptr[kcl + r + 1], kcl, j0 + k, Z + (int64_t)k * kcl);
}

extern "C" void schur_branch_rhs_host(int32_t kcl, int32_t m, const int32_t* indptr, const int32_t* indices,
                                      const double* data, const double* r, const double* t, double* out) {
    for (int32_t q = 0; q < m; ++q)
        out[q] = schur_branch_rhs(indices, data, indptr[kcl + q], indptr[kcl + q + 1], kcl, r[kcl + q], t);
}

extern "C" void schur_node_rhs_host(int32_t kcl, const int32_t* b_ptr, const int32_t* b_col, const double* b_val,
                                    const double* r, const double* xb, double* out) {
    for (int32_t i = 0; i < kcl; ++i) out[i] = schur_node_rhs(b_col, b_val, b_ptr[i], b_ptr[i + 1], r[i], xb);
}

extern "C" void schur_residual_host(int32_t n, const int32_t* indptr, const int32_t* indices, const double* data,
                                    const double* rhs, const double* x, double* r) {
    for (int32_t i = 0; i < n; ++i) r[i] = schur_branch_rhs(indices, data, indptr[i], indptr[i + 1], n, rhs[i], x);
}
