// Arithmetic of the AMG V-cycle's vector steps, written once for the CUDA kernels (amg_kernels.cuh)
// and for the host harness the CPU tests compile with g++ -ffp-contract=off
// (tests/host_check/amg_cycle_host.cpp).  Every rounding step is explicit, so the fused sweeps,
// which form x0 and the prolongated iterate at every gathered column, compute bit for bit what the
// unfused kernels store and read back, whatever the compiler would contract on its own.
#pragma once

#if defined(__CUDACC__)
#define AMGC_HD __host__ __device__ __forceinline__
#else
#include <cmath>
#define AMGC_HD static inline
#endif

#if defined(__CUDA_ARCH__)
#define AMGC_MUL(a, b) __dmul_rn(a, b)
#define AMGC_SUB(a, b) __dsub_rn(a, b)
#define AMGC_FMA(a, b, c) __fma_rn(a, b, c)
#else
#define AMGC_MUL(a, b) ((a) * (b))
#define AMGC_SUB(a, b) ((a) - (b))
#define AMGC_FMA(a, b, c) std::fma(a, b, c)
#endif

// One entry of a row product: acc + a_ij x_j, one rounding (the CSR-order FMA chain of sell_row_dot).
AMGC_HD double amg_dot_step(double a, double x, double acc) { return AMGC_FMA(a, x, acc); }

// Jacobi start from a zero guess: x0 = (omega d) b, d = 1 / a_ii.
AMGC_HD double amg_jacobi_start(double omega, double dinv, double b) {
    return AMGC_MUL(AMGC_MUL(omega, dinv), b);
}

// Coarse correction: x~ = x0 + scale xc[agg], one rounding.
AMGC_HD double amg_prolong_add(double scale, double xc, double x0) { return AMGC_FMA(scale, xc, x0); }

// Residual r = b - (A x)_i.
AMGC_HD double amg_residual(double b, double acc) { return AMGC_SUB(b, acc); }

// Damped Jacobi sweep: y = x + (omega d)(b - (A x)_i), one rounding for the update.
AMGC_HD double amg_jacobi_update(double omega, double dinv, double b, double acc, double x) {
    return AMGC_FMA(AMGC_MUL(omega, dinv), AMGC_SUB(b, acc), x);
}
