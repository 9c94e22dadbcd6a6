// Per-row rules of the Schur-complement solve (csrc/schur.cu), written once as __host__ __device__
// functions so the GPU kernels and the CPU-side check (tests/host_check/schur_host.cpp against
// tests/schur_mirror.py) share them.
//
// The MNA matrix with sorted columns is G = [[L, B], [C, D]]: rows and columns 0..kcl-1 are the
// node rows, kcl..n-1 the branch rows.  Only resistors stamp into the node-node block, so L is the
// resistor Laplacian; B (node rows, branch columns) and C | D (the branch rows) hold every source
// stamp.  In a node row the L entries are the prefix with column < kcl and the B entries the suffix.
//
// Every sum runs over the entries of one row in CSR order, a rounded product then a rounded add per
// entry (no contraction), then one subtraction: the same bits on the device, on the host and in numpy.
#pragma once
#include <stdint.h>

#ifndef __CUDACC__
#define __host__
#define __device__
#endif

#ifdef __CUDA_ARCH__
__device__ __forceinline__ double schur_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double schur_add(double a, double b) { return __dadd_rn(a, b); }
#else
inline double schur_mul(double a, double b) { return a * b; }   // compiled with -ffp-contract=off
inline double schur_add(double a, double b) { return a + b; }
#endif

// number of L entries of a node row (the prefix of its sorted columns below kcl)
__host__ __device__ inline int32_t schur_l_count(const int32_t* indices, int64_t begin, int64_t end, int32_t kcl) {
    int32_t c = 0;
    for (int64_t p = begin; p < end && indices[p] < kcl; ++p) ++c;
    return c;
}

// sum over the entries of [begin, end) with column < kcl of value * z[column], in order
__host__ __device__ inline double schur_row_dot_nodes(const int32_t* indices, const double* data, int64_t begin,
                                                      int64_t end, int32_t kcl, const double* z) {
    double acc = 0.0;
    for (int64_t p = begin; p < end; ++p) {
        const int32_t c = indices[p];
        if (c < kcl) acc = schur_add(acc, schur_mul(data[p], z[c]));
    }
    return acc;
}

// S[r, j] = D[r, j] - (C z)[r] for the branch row r = [begin, end) of G and branch column j; z is the
// column j of L^-1 B
__host__ __device__ inline double schur_column_entry(const int32_t* indices, const double* data, int64_t begin,
                                                     int64_t end, int32_t kcl, int32_t j, const double* z) {
    double d = 0.0;
    for (int64_t p = begin; p < end; ++p)
        if (indices[p] == kcl + j) d = data[p];
    return d - schur_row_dot_nodes(indices, data, begin, end, kcl, z);
}

// r_b - C t for one branch row
__host__ __device__ inline double schur_branch_rhs(const int32_t* indices, const double* data, int64_t begin,
                                                   int64_t end, int32_t kcl, double rb, const double* t) {
    return rb - schur_row_dot_nodes(indices, data, begin, end, kcl, t);
}

// r_n - B x_b for one node row; bcol / bval: the row's B entries (branch index, value), in order
__host__ __device__ inline double schur_node_rhs(const int32_t* bcol, const double* bval, int64_t begin, int64_t end,
                                                 double rn, const double* xb) {
    double acc = 0.0;
    for (int64_t p = begin; p < end; ++p) acc = schur_add(acc, schur_mul(bval[p], xb[bcol[p]]));
    return rn - acc;
}
