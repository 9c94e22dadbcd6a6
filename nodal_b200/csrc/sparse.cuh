// Sparse matrix formats shared by the Krylov solvers.
#pragma once
#include "common.cuh"

// Sliced ELLPACK, slice height 32 (one warp per slice, one lane per row).  Entry k of
// the row handled by lane l of slice s lives at slice_off[s] + k*32 + l, so every load
// of a warp is one fully coalesced 128-B (cols) / 256-B (vals) request.  Rows are kept
// in their original order and columns in CSR order, so the per-row summation order is
// the CSR one.  Padding entries have val 0 and col = the row itself.
struct nodal_sell {
    nodal_ctx* ctx = nullptr;   // owner of the buffers (pool)
    int device = 0;
    int32_t n = 0;
    int32_t nslices = 0;
    int64_t padded = 0;        // stored entries (incl. padding)
    int64_t nnz = 0;
    u32* slice_w = nullptr;    // [nslices + 1]: exclusive scan of slice widths (units: k-steps)
    int32_t* cols = nullptr;   // [padded]  (second half of the vals block)
    double* vals = nullptr;    // [padded]
    size_t store_bytes = 0;    // bytes of the [vals | cols] block
    double* dinv = nullptr;    // [n] 1 / diagonal (1 where the diagonal is 0)
};

int sell_from_csr(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                  const int32_t* indices, const double* data, nodal_sell** out, cudaStream_t st,
                  const double* sc = nullptr);   // sc: optional row/column scale factors (S A S)
void sell_free(nodal_sell* m);
int sell_set_l2_window(nodal_ctx* ctx, const nodal_sell* m, cudaStream_t st);   // see spmv.cu
void sell_clear_l2_window(cudaStream_t st);

// y = A x on the generic CSR path
int csr_spmv_launch(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                    const int32_t* indices, const double* data, const double* x, double* y,
                    cudaStream_t st);
// The same for `rows` rows of a larger matrix (shape_n rows, shape_nnz entries): the lanes per row
// follow the whole matrix's shape, so every row's sum is formed as csr_spmv_launch forms it there.
int csr_spmv_rows_launch(nodal_ctx* ctx, int32_t rows, const int32_t* indptr, const int32_t* indices,
                         const double* data, const double* x, double* y, int32_t shape_n, int64_t shape_nnz,
                         cudaStream_t st);

#ifdef __CUDACC__
#include "amg_cycle_core.cuh"

// The operand of a row product at column c: here a stored vector.  The fused V-cycle sweeps
// (amg_kernels.cuh) pass functors that form the operand from other vectors instead.
struct SellLoad {
    const double* __restrict__ x;
    __device__ __forceinline__ double operator()(int32_t c) const { return __ldg(&x[c]); }
};

// Dot product of one SELL row (lane) with the gathered operand: entries k = 0..w-1 at base + 32k.
// Straight-line code per width -- all column/value loads first, then all gathers, then the FMA
// chain in CSR order -- so the memory-level parallelism does not depend on how the compiler treats
// a predicated unrolled loop (it silently fell back to a rolled, dependent loop in one kernel).
template <int W, class G>
__device__ __forceinline__ double sell_dot_fixed(const int32_t* __restrict__ cols,
                                                 const double* __restrict__ vals, int64_t base,
                                                 const G& gather, double acc) {
    int32_t c[W];
    double v[W], xv[W];
#pragma unroll
    for (int i = 0; i < W; ++i) {
        c[i] = cols[base + (int64_t)i * 32];
        v[i] = vals[base + (int64_t)i * 32];
    }
#pragma unroll
    for (int i = 0; i < W; ++i) xv[i] = gather(c[i]);
#pragma unroll
    for (int i = 0; i < W; ++i) acc = amg_dot_step(v[i], xv[i], acc);
    return acc;
}

template <class G>
__device__ __forceinline__ double sell_row_gather(const int32_t* __restrict__ cols,
                                                  const double* __restrict__ vals, int64_t base, int w,
                                                  const G& x) {
    double acc = 0.0;
    int k = 0;
    for (; k + 8 <= w; k += 8) acc = sell_dot_fixed<8>(cols, vals, base + (int64_t)k * 32, x, acc);
    const int64_t b = base + (int64_t)k * 32;
    switch (w - k) {   // warp-uniform
        case 7: acc = sell_dot_fixed<7>(cols, vals, b, x, acc); break;
        case 6: acc = sell_dot_fixed<6>(cols, vals, b, x, acc); break;
        case 5: acc = sell_dot_fixed<5>(cols, vals, b, x, acc); break;
        case 4: acc = sell_dot_fixed<4>(cols, vals, b, x, acc); break;
        case 3: acc = sell_dot_fixed<3>(cols, vals, b, x, acc); break;
        case 2: acc = sell_dot_fixed<2>(cols, vals, b, x, acc); break;
        case 1: acc = sell_dot_fixed<1>(cols, vals, b, x, acc); break;
        default: break;
    }
    return acc;
}

__device__ __forceinline__ double sell_row_dot(const int32_t* __restrict__ cols,
                                               const double* __restrict__ vals, int64_t base, int w,
                                               const double* __restrict__ x) {
    return sell_row_gather(cols, vals, base, w, SellLoad{x});
}
#endif
