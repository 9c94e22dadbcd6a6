// Schur complement of the branch rows of an MNA system, for netlists with op-amps and dependent
// sources (nodal_b200/schur.py; tests/schur_mirror.py states the algorithm in numpy).  With the
// sorted MNA matrix G = [[L, B], [C, D]] (L the resistor Laplacian of the kcl node rows):
//
//   nodal_schur_split_scan / _place   L as its own CSR and B as per-row lists (branch index, value),
//                                     by count / scan / copy of the node rows of G; C | D are the
//                                     branch rows of G, used in place.
//   nodal_schur_rhs_batch             the (K, kcl) right-hand side of the branch columns [j0, j0 + K)
//                                     of B, for one batched AMG solve (csrc/amg_multi.cu).
//   nodal_schur_columns               S[:, j0 : j0 + K] = D - C Z from the batch's solutions Z.
//   nodal_schur_branch_rhs / _node_rhs  r_b - C t and r_n - B x_b: the two couplings of one application
//                                     of the block inverse.
//   nodal_schur_residual / _add       r = rhs - G x with its norms, and x += d: the refinement steps.
//
// The per-row rules are in schur_core.cuh.  One thread owns each output entry and sums its row in
// CSR order; nothing accumulates floating-point values with atomics, so results are bitwise
// reproducible.
#include "common.cuh"
#include "schur_core.cuh"

constexpr int SC = 256;

static int sc_grid(nodal_ctx* ctx, int64_t work) {
    int64_t g = (work + SC - 1) / SC;
    const int64_t cap = (int64_t)ctx->num_sms * 16;
    return (int)(g < 1 ? 1 : g < cap ? g : cap);
}

#define GRID_STRIDE(i, count) \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (count); i += (int64_t)gridDim.x * blockDim.x)

__global__ void __launch_bounds__(SC)
schur_count_kernel(int32_t kcl, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                   u32* __restrict__ lcount, u32* __restrict__ bcount) {
    GRID_STRIDE(i, kcl) {
        const int32_t l = schur_l_count(indices, indptr[i], indptr[i + 1], kcl);
        lcount[i] = (u32)l;
        bcount[i] = (u32)(indptr[i + 1] - indptr[i] - l);
    }
}

__global__ void __launch_bounds__(SC)
schur_place_kernel(int32_t kcl, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                   const double* __restrict__ data, const int32_t* __restrict__ l_ptr, int32_t* __restrict__ l_idx,
                   double* __restrict__ l_val, const int32_t* __restrict__ b_ptr, int32_t* __restrict__ b_col,
                   double* __restrict__ b_val) {
    GRID_STRIDE(i, kcl) {
        const int32_t p0 = indptr[i], nl = l_ptr[i + 1] - l_ptr[i];
        for (int32_t q = 0; q < nl; ++q) {
            l_idx[l_ptr[i] + q] = indices[p0 + q];
            l_val[l_ptr[i] + q] = data[p0 + q];
        }
        for (int32_t q = 0; q < b_ptr[i + 1] - b_ptr[i]; ++q) {
            b_col[b_ptr[i] + q] = indices[p0 + nl + q] - kcl;
            b_val[b_ptr[i] + q] = data[p0 + nl + q];
        }
    }
}

__global__ void __launch_bounds__(SC)
schur_rhs_batch_kernel(int32_t kcl, int32_t j0, int32_t K, const int32_t* __restrict__ b_ptr,
                       const int32_t* __restrict__ b_col, const double* __restrict__ b_val, double* __restrict__ rhs) {
    GRID_STRIDE(i, kcl) {
        for (int32_t k = 0; k < K; ++k) rhs[(int64_t)k * kcl + i] = 0.0;
        for (int32_t p = b_ptr[i]; p < b_ptr[i + 1]; ++p) {
            const int32_t k = b_col[p] - j0;
            if (k >= 0 && k < K) rhs[(int64_t)k * kcl + i] = b_val[p];
        }
    }
}

__global__ void __launch_bounds__(SC)
schur_columns_kernel(int32_t kcl, int32_t m, int32_t j0, int32_t K, const int32_t* __restrict__ indptr,
                     const int32_t* __restrict__ indices, const double* __restrict__ data, const double* __restrict__ Z,
                     double* __restrict__ S) {
    GRID_STRIDE(e, (int64_t)m * K) {
        const int32_t r = (int32_t)(e / K), k = (int32_t)(e - (int64_t)r * K);
        S[(int64_t)r * m + j0 + k] = schur_column_entry(indices, data, indptr[kcl + r], indptr[kcl + r + 1], kcl, j0 + k,
                                                        Z + (int64_t)k * kcl);
    }
}

__global__ void __launch_bounds__(SC)
schur_branch_rhs_kernel(int32_t kcl, int32_t m, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                        const double* __restrict__ data, const double* __restrict__ r, const double* __restrict__ t,
                        double* __restrict__ out) {
    GRID_STRIDE(q, m) {
        const int64_t row = kcl + q;
        out[q] = schur_branch_rhs(indices, data, indptr[row], indptr[row + 1], kcl, r[row], t);
    }
}

__global__ void __launch_bounds__(SC)
schur_node_rhs_kernel(int32_t kcl, const int32_t* __restrict__ b_ptr, const int32_t* __restrict__ b_col,
                      const double* __restrict__ b_val, const double* __restrict__ r, const double* __restrict__ xb,
                      double* __restrict__ out) {
    GRID_STRIDE(i, kcl) out[i] = schur_node_rhs(b_col, b_val, b_ptr[i], b_ptr[i + 1], r[i], xb);
}

// r = rhs - G x (every column counts as a "node" column: kcl = n), block partials of sum r^2, sum rhs^2
__global__ void __launch_bounds__(SC)
schur_residual_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                      const double* __restrict__ data, const double* __restrict__ rhs, const double* __restrict__ x,
                      double* __restrict__ r, double* __restrict__ part) {
    __shared__ double smem[33];
    double rr = 0.0, bb = 0.0;
    GRID_STRIDE(i, n) {
        const double b = rhs[i];
        const double v = schur_branch_rhs(indices, data, indptr[i], indptr[i + 1], n, b, x);
        r[i] = v;
        rr = __dadd_rn(rr, __dmul_rn(v, v));
        bb = __dadd_rn(bb, __dmul_rn(b, b));
    }
    rr = block_sum(rr, smem);
    bb = block_sum(bb, smem);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = rr;
        part[gridDim.x + blockIdx.x] = bb;
    }
}

__global__ void __launch_bounds__(SC)
schur_norms_kernel(int32_t nblocks, const double* __restrict__ part, double* __restrict__ sums) {
    __shared__ double smem[33];
    const double rr = reduce_partials(part, nblocks, smem);
    const double bb = reduce_partials(part + nblocks, nblocks, smem);
    if (threadIdx.x == 0) { sums[0] = rr; sums[1] = bb; }
}

__global__ void __launch_bounds__(SC)
schur_add_kernel(int64_t count, double* __restrict__ x, const double* __restrict__ d) {
    GRID_STRIDE(i, count) x[i] = __dadd_rn(x[i], d[i]);
}

extern "C" int nodal_schur_split_scan(nodal_ctx* ctx, int32_t kcl, const int32_t* indptr, const int32_t* indices,
                                      int32_t* l_ptr, int32_t* b_ptr, int64_t* nnz_h, void* stream) {
    if (!ctx || kcl < 0 || !indptr || !l_ptr || !b_ptr || !nnz_h) return NODAL_BAD_ARG;
    NvtxRange nvtx_range("nodal_schur_split_scan");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t count = (int64_t)kcl + 1;
    NODAL_TRY(ctx_reserve(ctx, 2 * scan_scratch_bytes(count) + 4096));
    u32* totals = carve<u32>(ctx, 2);
    if (!totals) return NODAL_CUDA_ERROR;
    u32* lc = reinterpret_cast<u32*>(l_ptr);
    u32* bc = reinterpret_cast<u32*>(b_ptr);
    CUDA_TRY(cudaMemsetAsync(lc + kcl, 0, sizeof(u32), st));
    CUDA_TRY(cudaMemsetAsync(bc + kcl, 0, sizeof(u32), st));
    if (kcl > 0) {
        schur_count_kernel<<<sc_grid(ctx, kcl), SC, 0, st>>>(kcl, indptr, indices, lc, bc);
        KERNEL_CHECK();
    }
    NODAL_TRY(scan_exclusive_u32(ctx, lc, lc, count, totals, st));
    NODAL_TRY(scan_exclusive_u32(ctx, bc, bc, count, totals + 1, st));
    u32* host = reinterpret_cast<u32*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(host, totals, 2 * sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    nnz_h[0] = host[0];
    nnz_h[1] = host[1];
    return NODAL_OK;
}

extern "C" int nodal_schur_split_place(nodal_ctx* ctx, int32_t kcl, const int32_t* indptr, const int32_t* indices,
                                       const double* data, const int32_t* l_ptr, int32_t* l_idx, double* l_val,
                                       const int32_t* b_ptr, int32_t* b_col, double* b_val, void* stream) {
    if (!ctx || kcl < 0) return NODAL_BAD_ARG;
    if (kcl == 0) return NODAL_OK;
    NvtxRange nvtx_range("nodal_schur_split_place");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_place_kernel<<<sc_grid(ctx, kcl), SC, 0, st>>>(kcl, indptr, indices, data, l_ptr, l_idx, l_val, b_ptr, b_col,
                                                        b_val);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_schur_rhs_batch(nodal_ctx* ctx, int32_t kcl, int32_t j0, int32_t K, const int32_t* b_ptr,
                                     const int32_t* b_col, const double* b_val, double* rhs, void* stream) {
    if (!ctx || kcl < 0 || K < 1 || j0 < 0) return NODAL_BAD_ARG;
    if (kcl == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_rhs_batch_kernel<<<sc_grid(ctx, kcl), SC, 0, st>>>(kcl, j0, K, b_ptr, b_col, b_val, rhs);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_schur_columns(nodal_ctx* ctx, int32_t kcl, int32_t m, int32_t j0, int32_t K, const int32_t* indptr,
                                   const int32_t* indices, const double* data, const double* Z, double* S,
                                   void* stream) {
    if (!ctx || kcl < 0 || m < 0 || K < 1 || j0 < 0 || j0 + K > m) return NODAL_BAD_ARG;
    if (m == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_columns_kernel<<<sc_grid(ctx, (int64_t)m * K), SC, 0, st>>>(kcl, m, j0, K, indptr, indices, data, Z, S);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_schur_branch_rhs(nodal_ctx* ctx, int32_t kcl, int32_t m, const int32_t* indptr,
                                      const int32_t* indices, const double* data, const double* r, const double* t,
                                      double* out, void* stream) {
    if (!ctx || kcl < 0 || m < 0) return NODAL_BAD_ARG;
    if (m == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_branch_rhs_kernel<<<sc_grid(ctx, m), SC, 0, st>>>(kcl, m, indptr, indices, data, r, t, out);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_schur_node_rhs(nodal_ctx* ctx, int32_t kcl, const int32_t* b_ptr, const int32_t* b_col,
                                    const double* b_val, const double* r, const double* xb, double* out, void* stream) {
    if (!ctx || kcl < 0) return NODAL_BAD_ARG;
    if (kcl == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_node_rhs_kernel<<<sc_grid(ctx, kcl), SC, 0, st>>>(kcl, b_ptr, b_col, b_val, r, xb, out);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_schur_residual(nodal_ctx* ctx, int32_t n, const int32_t* indptr, const int32_t* indices,
                                    const double* data, const double* rhs, const double* x, double* r, double* sums_h,
                                    void* stream) {
    if (!ctx || n < 0 || !sums_h) return NODAL_BAD_ARG;
    sums_h[0] = sums_h[1] = 0.0;
    if (n == 0) return NODAL_OK;
    NvtxRange nvtx_range("nodal_schur_residual");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int grid = sc_grid(ctx, n);
    NODAL_TRY(ctx_reserve(ctx, sizeof(double) * (2 * (size_t)grid + 2) + 1024));
    double* part = carve<double>(ctx, 2 * (size_t)grid);
    double* sums = carve<double>(ctx, 2);
    if (!part || !sums) return NODAL_CUDA_ERROR;
    schur_residual_kernel<<<grid, SC, 0, st>>>(n, indptr, indices, data, rhs, x, r, part);
    KERNEL_CHECK();
    schur_norms_kernel<<<1, SC, 0, st>>>(grid, part, sums);
    KERNEL_CHECK();
    double* host = reinterpret_cast<double*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(host, sums, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    sums_h[0] = host[0];
    sums_h[1] = host[1];
    return NODAL_OK;
}

extern "C" int nodal_schur_add(nodal_ctx* ctx, int64_t count, double* x, const double* d, void* stream) {
    if (!ctx || count < 0) return NODAL_BAD_ARG;
    if (count == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    schur_add_kernel<<<sc_grid(ctx, count), SC, 0, st>>>(count, x, d);
    KERNEL_CHECK();
    return NODAL_OK;
}
