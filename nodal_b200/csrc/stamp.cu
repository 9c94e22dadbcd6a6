// Stamping kernel: struct-of-arrays component table -> keyed COO triples.
// Replaces the Python loop of Circuit.build_model (nodal/nodal.py:357-390).
//
// One thread per component.  Table columns are read coalesced (33 B/component); the
// `stride` output slots of a warp's 32 components form one contiguous 32*stride*8-byte
// span in keys[] and vals[], which is staged through shared memory so the global
// stores are fully coalesced 8-byte-per-lane writes.
#include <algorithm>

#include "common.cuh"
#include "stamp_core.cuh"

constexpr int STAMP_THREADS = 256;

template <int STRIDE>
__global__ void __launch_bounds__(STAMP_THREADS)
stamp_coo_kernel(int64_t ncomp, const uint8_t* __restrict__ type, const double* __restrict__ value,
                 const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                 const int32_t* __restrict__ c, const int32_t* __restrict__ d,
                 const int32_t* __restrict__ drv, const int32_t* __restrict__ branch,
                 int32_t kcl, int32_t n, int32_t colbits,
                 u64* __restrict__ keys, double* __restrict__ vals) {
    __shared__ u64 s_key[STAMP_THREADS * STRIDE];
    __shared__ double s_val[STAMP_THREADS * STRIDE];
    const u64 invalid = (u64)(u32)n << colbits;
    const int64_t tiles = (ncomp + STAMP_THREADS - 1) / STAMP_THREADS;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * STAMP_THREADS;
        const int64_t i = base + threadIdx.x;
        StampOut o;
        o.count = 0;
        if (i < ncomp) {
            const int t = type[i];
            double dv = 1.0;
            if ((t == NODAL_T_CCVS || t == NODAL_T_CCCS) && drv) dv = value[drv[i]];
            // c / d / drv / branch may be null for R / A-only tables (the columns hold constants
            // then and are neither uploaded nor read: 17 instead of 33 bytes per component)
            stamp_component(t, value[i], a[i], b[i], c ? c[i] : -2, d ? d[i] : -2, dv, branch ? branch[i] : -1, kcl, n, o);
        }
#pragma unroll
        for (int k = 0; k < STRIDE; ++k) {
            const bool live = k < o.count;
            s_key[threadIdx.x * STRIDE + k] =
                live ? (((u64)(u32)o.row[k] << colbits) | (u64)(u32)o.col[k]) : invalid;
            s_val[threadIdx.x * STRIDE + k] = live ? o.val[k] : 0.0;
        }
        __syncthreads();
        const int64_t out0 = base * STRIDE;
        const int64_t lim = ((ncomp - base < STAMP_THREADS) ? (ncomp - base) : (int64_t)STAMP_THREADS) * STRIDE;
        for (int64_t j = threadIdx.x; j < lim; j += STAMP_THREADS) {
            keys[out0 + j] = s_key[j];
            vals[out0 + j] = s_val[j];
        }
        __syncthreads();
    }
}

extern "C" int nodal_stamp_coo(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type,
                               const double* value, const int32_t* a, const int32_t* b,
                               const int32_t* c, const int32_t* d, const int32_t* drv,
                               const int32_t* branch, int32_t kcl, int32_t n, int32_t stride,
                               int32_t colbits, uint64_t* keys, double* vals, void* stream) {
    NvtxRange nvtx_range("nodal_stamp_coo");
    if (!ctx || ncomp < 0 || n < 0 || kcl > n) return NODAL_BAD_ARG;
    if (colbits < 1 || colbits > 31 || ((int64_t)n >> colbits) != 0) {
        nodal_set_error("nodal_stamp_coo: colbits=%d cannot hold column index n=%d", colbits, n);
        return NODAL_BAD_ARG;
    }
    if (ncomp == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t tiles = (ncomp + STAMP_THREADS - 1) / STAMP_THREADS;
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)ctx->num_sms * 8);
    u64* k64 = reinterpret_cast<u64*>(keys);
#define LAUNCH(S)                                                                              \
    stamp_coo_kernel<S><<<grid, STAMP_THREADS, 0, st>>>(ncomp, type, value, a, b, c, d, drv,   \
                                                        branch, kcl, n, colbits, k64, vals)
    switch (stride) {
        case 2: LAUNCH(2); break;
        case 4: LAUNCH(4); break;
        case 5: LAUNCH(5); break;
        case 6: LAUNCH(6); break;
        default:
            nodal_set_error("nodal_stamp_coo: stride must be 2, 4, 5 or 6 (got %d)", stride);
            return NODAL_BAD_ARG;
    }
#undef LAUNCH
    KERNEL_CHECK();
    return NODAL_OK;
}

// ---------------------------------------------------------------- row-partitioned assembly
// A rank of the multi-GPU path stamps only the components that write one of its rows [rb, re)
// (global stamping order kept, so its rows of G are bit-identical to the single-GPU CSR).  The
// selection runs on the device: flags -> exclusive scan -> ordered gather of the eight columns.
// A component is selected when a lead is on a row in [rb, re) -- the only rows an R / A component
// writes -- or when the kernel's extra test holds:
//   NoExtra        nothing more (R / A tables)
//   OwnBranchRow   an E row whose branch row kcl + branch is in [rb, re) (R / A / E tables)
//   TypeIs         components of one type, with an empty [rb, re) (the E rows of the source forest)
struct NoExtra {
    __device__ __forceinline__ bool operator()(int64_t, int32_t, int32_t) const { return false; }
};

struct OwnBranchRow {
    const uint8_t* __restrict__ type;
    const int32_t* __restrict__ branch;
    int32_t kcl;
    __device__ __forceinline__ bool operator()(int64_t i, int32_t rb, int32_t re) const {
        if (type[i] != NODAL_T_E) return false;
        const int32_t r = kcl + branch[i];
        return r >= rb && r < re;
    }
};

struct TypeIs {
    const uint8_t* __restrict__ type;
    int32_t t;
    __device__ __forceinline__ bool operator()(int64_t i, int32_t, int32_t) const { return type[i] == t; }
};

template <class Extra>
__global__ void __launch_bounds__(STAMP_THREADS)
select_flag_kernel(int64_t ncomp, const int32_t* __restrict__ a, const int32_t* __restrict__ b, int32_t rb,
                   int32_t re, u32* __restrict__ flag, Extra extra) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncomp; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t x = a[i], y = b[i];
        flag[i] = ((x >= rb && x < re) || (y >= rb && y < re) || extra(i, rb, re)) ? 1u : 0u;
    }
}

template <class Extra>
__global__ void __launch_bounds__(STAMP_THREADS)
select_gather_kernel(int64_t ncomp, const u32* __restrict__ pos, int32_t rb, int32_t re,
                     const uint8_t* __restrict__ type, const double* __restrict__ value,
                     const int32_t* __restrict__ a, const int32_t* __restrict__ b, const int32_t* __restrict__ c,
                     const int32_t* __restrict__ d, const int32_t* __restrict__ drv, const int32_t* __restrict__ branch,
                     uint8_t* __restrict__ o_type, double* __restrict__ o_value, int32_t* __restrict__ o_a,
                     int32_t* __restrict__ o_b, int32_t* __restrict__ o_c, int32_t* __restrict__ o_d,
                     int32_t* __restrict__ o_drv, int32_t* __restrict__ o_branch, Extra extra) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncomp; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t x = a[i], y = b[i];
        if (!((x >= rb && x < re) || (y >= rb && y < re) || extra(i, rb, re))) continue;
        const u32 p = pos[i];
        o_type[p] = type[i]; o_value[p] = value[i]; o_a[p] = x; o_b[p] = y;
        if (c) o_c[p] = c[i];
        if (d) o_d[p] = d[i];
        if (drv) o_drv[p] = drv[i];
        if (branch) o_branch[p] = branch[i];
    }
}

static int select_grid(nodal_ctx* ctx, int64_t ncomp) {
    return (int)std::min<int64_t>((ncomp + STAMP_THREADS - 1) / STAMP_THREADS, (int64_t)ctx->num_sms * 16);
}

template <class Extra>
static int select_scan(nodal_ctx* ctx, int64_t ncomp, const int32_t* a, const int32_t* b, int32_t rb, int32_t re,
                       Extra extra, uint32_t* pos, int64_t* count_h, void* stream) {
    if (!ctx || ncomp < 0 || !count_h || ncomp >= ((int64_t)1 << 32)) return NODAL_BAD_ARG;
    *count_h = 0;
    if (ncomp == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes(ncomp) + 4096));
    u32* total = carve<u32>(ctx, 16);
    if (!total) return NODAL_CUDA_ERROR;
    select_flag_kernel<Extra><<<select_grid(ctx, ncomp), STAMP_THREADS, 0, st>>>(ncomp, a, b, rb, re, pos, extra);
    KERNEL_CHECK();
    NODAL_TRY(scan_exclusive_u32(ctx, pos, pos, ncomp, total, st));
    u32* total_h = reinterpret_cast<u32*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(total_h, total, sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *count_h = total_h[0];
    return NODAL_OK;
}

template <class Extra>
static int select_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t rb, int32_t re, Extra extra,
                         const uint8_t* type,
                         const double* value, const int32_t* a, const int32_t* b, const int32_t* c, const int32_t* d,
                         const int32_t* drv, const int32_t* branch, uint8_t* o_type, double* o_value, int32_t* o_a,
                         int32_t* o_b, int32_t* o_c, int32_t* o_d, int32_t* o_drv, int32_t* o_branch, void* stream) {
    if (!ctx || ncomp < 0) return NODAL_BAD_ARG;
    if (ncomp == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    select_gather_kernel<Extra><<<select_grid(ctx, ncomp), STAMP_THREADS, 0, st>>>(
        ncomp, pos, rb, re, type, value, a, b, c, d, drv, branch, o_type, o_value, o_a, o_b, o_c, o_d, o_drv, o_branch,
        extra);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_table_select_scan(nodal_ctx* ctx, int64_t ncomp, const int32_t* a, const int32_t* b,
                                       int32_t rb, int32_t re, uint32_t* pos, int64_t* count_h, void* stream) {
    return select_scan(ctx, ncomp, a, b, rb, re, NoExtra{}, pos, count_h, stream);
}

extern "C" int nodal_table_select_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t rb, int32_t re,
                                         const uint8_t* type, const double* value, const int32_t* a,
                                         const int32_t* b, const int32_t* c, const int32_t* d, const int32_t* drv,
                                         const int32_t* branch, uint8_t* o_type, double* o_value, int32_t* o_a,
                                         int32_t* o_b, int32_t* o_c, int32_t* o_d, int32_t* o_drv,
                                         int32_t* o_branch, void* stream) {
    return select_gather(ctx, ncomp, pos, rb, re, NoExtra{}, type, value, a, b, c, d, drv, branch, o_type, o_value,
                         o_a, o_b, o_c, o_d, o_drv, o_branch, stream);
}

extern "C" int nodal_table_select_mna_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                                           const int32_t* b, const int32_t* branch, int32_t kcl, int32_t rb,
                                           int32_t re, uint32_t* pos, int64_t* count_h, void* stream) {
    if (ncomp > 0 && (!type || !branch)) return NODAL_BAD_ARG;
    return select_scan(ctx, ncomp, a, b, rb, re, OwnBranchRow{type, branch, kcl}, pos, count_h, stream);
}

extern "C" int nodal_table_select_mna_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t kcl,
                                             int32_t rb, int32_t re, const uint8_t* type, const double* value,
                                             const int32_t* a, const int32_t* b, const int32_t* c, const int32_t* d,
                                             const int32_t* drv, const int32_t* branch, uint8_t* o_type,
                                             double* o_value, int32_t* o_a, int32_t* o_b, int32_t* o_c, int32_t* o_d,
                                             int32_t* o_drv, int32_t* o_branch, void* stream) {
    if (ncomp > 0 && (!type || !branch)) return NODAL_BAD_ARG;
    return select_gather(ctx, ncomp, pos, rb, re, OwnBranchRow{type, branch, kcl}, type, value, a, b, c, d, drv,
                         branch, o_type, o_value, o_a, o_b, o_c, o_d, o_drv, o_branch, stream);
}

extern "C" int nodal_table_select_type_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                                            const int32_t* b, int32_t t, uint32_t* pos, int64_t* count_h,
                                            void* stream) {
    if (ncomp > 0 && !type) return NODAL_BAD_ARG;
    return select_scan(ctx, ncomp, a, b, 0, 0, TypeIs{type, t}, pos, count_h, stream);
}

extern "C" int nodal_table_select_type_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t t,
                                              const uint8_t* type, const double* value, const int32_t* a,
                                              const int32_t* b, const int32_t* c, const int32_t* d,
                                              const int32_t* drv, const int32_t* branch, uint8_t* o_type,
                                              double* o_value, int32_t* o_a, int32_t* o_b, int32_t* o_c,
                                              int32_t* o_d, int32_t* o_drv, int32_t* o_branch, void* stream) {
    if (ncomp > 0 && !type) return NODAL_BAD_ARG;
    return select_gather(ctx, ncomp, pos, 0, 0, TypeIs{type, t}, type, value, a, b, c, d, drv, branch, o_type, o_value,
                         o_a, o_b, o_c, o_d, o_drv, o_branch, stream);
}
