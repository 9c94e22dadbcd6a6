// TEST-ONLY: compiles the V-cycle arithmetic (nodal_b200/csrc/amg_cycle_core.cuh) for the CPU with
// g++ -ffp-contract=off and runs the steps of one level of the cycle on a CSR operator, in the
// unfused form (Jacobi start, residual sweep, prolongation, Jacobi sweep: each vector stored) and in
// the fused form of amg_cycle_sweep_kernel (x0 and the prolongated iterate formed at every gathered
// column), so `pytest -m "not gpu"` can check that the two forms agree bit for bit.  Row products
// are the FMA chain in CSR order, as sell_row_gather computes them.  Not part of the product library.
#include <stdint.h>

#include "../../nodal_b200/csrc/amg_cycle_core.cuh"

namespace {

template <class G>
double row_dot(const int32_t* indptr, const int32_t* indices, const double* data, int32_t i, const G& x) {
    double acc = 0.0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) acc = amg_dot_step(data[p], x(indices[p]), acc);
    return acc;
}

}  // namespace

// unfused: x = omega D^-1 b
extern "C" void amgc_jacobi0_host(int32_t n, const double* dinv, const double* b, double omega, double* x) {
    for (int32_t i = 0; i < n; ++i) x[i] = amg_jacobi_start(omega, dinv[i], b[i]);
}

// unfused: xa = x + scale xc[agg]
extern "C" void amgc_prolong_host(int32_t n, const int32_t* agg, const double* xc, double scale, const double* x,
                                  double* xa) {
    for (int32_t i = 0; i < n; ++i) xa[i] = amg_prolong_add(scale, xc[agg[i]], x[i]);
}

// unfused: mode 1 y = b - A x, mode 2 y = x + omega D^-1 (b - A x)
extern "C" void amgc_sweep_host(int32_t mode, int32_t n, const int32_t* indptr, const int32_t* indices,
                                const double* data, const double* dinv, const double* b, const double* x,
                                double omega, double* y) {
    auto gx = [&](int32_t c) { return x[c]; };
    for (int32_t i = 0; i < n; ++i) {
        const double acc = row_dot(indptr, indices, data, i, gx);
        y[i] = mode == 1 ? amg_residual(b[i], acc) : amg_jacobi_update(omega, dinv[i], b[i], acc, x[i]);
    }
}

// fused: mode 1 y = b - A x0, mode 2 y = x~ + omega D^-1 (b - A x~), x0 and x~ formed per column
extern "C" void amgc_fused_sweep_host(int32_t mode, int32_t n, const int32_t* indptr, const int32_t* indices,
                                      const double* data, const double* dinv, const double* b, double omega,
                                      const int32_t* agg, const double* xc, double scale, double* y) {
    auto x0 = [&](int32_t c) { return amg_jacobi_start(omega, dinv[c], b[c]); };
    auto xa = [&](int32_t c) { return amg_prolong_add(scale, xc[agg[c]], x0(c)); };
    for (int32_t i = 0; i < n; ++i) {
        if (mode == 1) y[i] = amg_residual(b[i], row_dot(indptr, indices, data, i, x0));
        else y[i] = amg_jacobi_update(omega, dinv[i], b[i], row_dot(indptr, indices, data, i, xa), xa(i));
    }
}

// bc[I] = sum of r over the members of aggregate I, in increasing row order (amg_restrict_kernel)
extern "C" void amgc_restrict_host(int32_t n, const int32_t* agg, const double* r, int32_t nc, double* bc) {
    for (int32_t I = 0; I < nc; ++I) bc[I] = 0.0;
    for (int32_t i = 0; i < n; ++i) bc[agg[i]] += r[i];
}
