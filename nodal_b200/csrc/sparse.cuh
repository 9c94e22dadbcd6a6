// Sparse matrix formats shared by the Krylov solvers.
#pragma once
#include "common.cuh"
#include "sell_core.cuh"

// Sliced ELLPACK, slice height 32 (one warp per slice, one lane per row).  Entry k of
// the row handled by lane l of slice s lives at slice_off[s] + k*32 + l, so every load
// of a warp is one fully coalesced request.  Rows are kept in their original order and columns
// in CSR order, so the per-row summation order is the CSR one.  Padding entries have val 0 and
// col = the row itself; the tail lanes of the last slice have col n - 1 (sell_core.cuh).
// Entries are stored in one of two encodings, chosen by sell_from_csr from the matrix:
//   compact  int16 col - row and a uint8 index into dict[ndict] (3 B per entry), when every offset
//            fits int16 and the values (with +0.0) have at most 256 distinct bit patterns;
//   wide     int32 col and double val (12 B per entry) otherwise, or with NODAL_SELL_WIDE=1.
// Readers go through sell_launch, which hands the kernel the view of the matrix's encoding.
struct nodal_sell {
    nodal_ctx* ctx = nullptr;   // owner of the buffers (pool)
    int device = 0;
    int32_t n = 0;
    int32_t nslices = 0;
    int64_t padded = 0;        // stored entries (incl. padding)
    int64_t nnz = 0;
    u32* slice_w = nullptr;    // [nslices + 1]: exclusive scan of slice widths (units: k-steps)
    bool compact = false;
    int32_t ndict = 0;         // compact: entries of dict
    void* store = nullptr;     // one block: wide [vals | cols], compact [dict | dcol | vidx]
    size_t store_bytes = 0;
    int32_t* cols = nullptr;   // wide: [padded]
    double* vals = nullptr;    // wide: [padded]
    double* dict = nullptr;    // compact: [SELL_DICT_MAX] values, sorted by bit pattern
    int16_t* dcol = nullptr;   // compact: [padded] col - row
    uint8_t* vidx = nullptr;   // compact: [padded] index into dict
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

// The two entry encodings as seen by a row product: load() reads the stored bytes of entry i,
// col() / val() decode them for row r (the lane's row, r >= n on tail lanes).
struct SellWide {
    const int32_t* __restrict__ cols;
    const double* __restrict__ vals;
    struct Entry { int32_t c; double v; };
    __device__ __forceinline__ Entry load(int64_t i) const { return {cols[i], vals[i]}; }
    __device__ __forceinline__ int32_t col(const Entry& e, int64_t) const { return e.c; }
    __device__ __forceinline__ double val(const Entry& e) const { return e.v; }
    __device__ __forceinline__ SellWide staged() const { return *this; }
};

// staged(), called by every thread of the block at the top of a reader kernel, returns the view the
// kernel reads through: for compact entries one with the 2 KB table copied to shared memory (measured
// faster than reading it through the read-only cache: post-smoothing sweep 0.2230 against 0.2316 ms at
// level 0 of the 4096^2 grid, profiles/r7_sell_table_shared_vs_ldg.json).
struct SellCompact {
    const int16_t* __restrict__ dcol;
    const uint8_t* __restrict__ vidx;
    const double* __restrict__ dict;
    struct Entry { int16_t d; uint8_t k; };
    __device__ __forceinline__ Entry load(int64_t i) const { return {dcol[i], vidx[i]}; }
    __device__ __forceinline__ int32_t col(const Entry& e, int64_t r) const { return sell_decode_col(e.d, r); }
    __device__ __forceinline__ double val(const Entry& e) const { return dict[e.k]; }
    __device__ __forceinline__ SellCompact staged() const {
        __shared__ double s[SELL_DICT_MAX];
        for (int i = threadIdx.x; i < SELL_DICT_MAX; i += blockDim.x) s[i] = __ldg(&dict[i]);
        __syncthreads();
        return {dcol, vidx, s};
    }
};

// Dot product of one SELL row (lane, row r) with the gathered operand: entries k = 0..w-1 at
// base + 32k.  Straight-line code per width -- all entry loads first, then all gathers (and table
// reads), then the FMA chain in CSR order -- so the memory-level parallelism does not depend on how
// the compiler treats a predicated unrolled loop (it silently fell back to a rolled, dependent loop
// in one kernel).
template <int W, class A, class G>
__device__ __forceinline__ double sell_dot_fixed(const A& a, int64_t base, int64_t r, const G& gather, double acc) {
    typename A::Entry e[W];
    double v[W], xv[W];
#pragma unroll
    for (int i = 0; i < W; ++i) e[i] = a.load(base + (int64_t)i * 32);
#pragma unroll
    for (int i = 0; i < W; ++i) {
        xv[i] = gather(a.col(e[i], r));
        v[i] = a.val(e[i]);
    }
#pragma unroll
    for (int i = 0; i < W; ++i) acc = amg_dot_step(v[i], xv[i], acc);
    return acc;
}

template <class A, class G>
__device__ __forceinline__ double sell_row_gather(const A& a, int64_t base, int64_t r, int w, const G& x) {
    double acc = 0.0;
    int k = 0;
    for (; k + 8 <= w; k += 8) acc = sell_dot_fixed<8>(a, base + (int64_t)k * 32, r, x, acc);
    const int64_t b = base + (int64_t)k * 32;
    switch (w - k) {   // warp-uniform
        case 7: acc = sell_dot_fixed<7>(a, b, r, x, acc); break;
        case 6: acc = sell_dot_fixed<6>(a, b, r, x, acc); break;
        case 5: acc = sell_dot_fixed<5>(a, b, r, x, acc); break;
        case 4: acc = sell_dot_fixed<4>(a, b, r, x, acc); break;
        case 3: acc = sell_dot_fixed<3>(a, b, r, x, acc); break;
        case 2: acc = sell_dot_fixed<2>(a, b, r, x, acc); break;
        case 1: acc = sell_dot_fixed<1>(a, b, r, x, acc); break;
        default: break;
    }
    return acc;
}

template <class A>
__device__ __forceinline__ double sell_row_dot(const A& a, int64_t base, int64_t r, int w,
                                               const double* __restrict__ x) {
    return sell_row_gather(a, base, r, w, SellLoad{x});
}

// Launches a SELL reader with the view of m's encoding: launch(view) is called with a SellWide or
// a SellCompact, and instantiates and launches the kernel for it.  No caller picks an encoding.
template <class L>
static inline void sell_launch(const nodal_sell* m, L&& launch) {
    if (m->compact) launch(SellCompact{m->dcol, m->vidx, m->dict});
    else launch(SellWide{m->cols, m->vals});
}
#endif
