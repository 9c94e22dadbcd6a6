// SpMV kernels: generic CSR (sub-warp per row) and the solver-private sliced-ELL format.
#include <algorithm>

#include "sparse.cuh"

constexpr int SPMV_THREADS = 256;

// ---------------------------------------------------------------- generic CSR
// TPR lanes cooperate on one row; a warp covers 32/TPR consecutive rows, i.e. one
// contiguous span of data[] / indices[].
template <int TPR>
__global__ void __launch_bounds__(SPMV_THREADS)
csr_spmv_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                const double* __restrict__ data, const double* __restrict__ x,
                double* __restrict__ y) {
    constexpr int RPW = 32 / TPR;
    const int lane = threadIdx.x & 31, sub = lane & (TPR - 1);
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r0 = warp * RPW; r0 < n; r0 += nwarps * RPW) {
        const int64_t row = r0 + lane / TPR;
        double acc = 0.0;
        if (row < n) {
            const int32_t e = indptr[row + 1];
            for (int32_t j = indptr[row] + sub; j < e; j += TPR)
                acc = fma(data[j], __ldg(&x[indices[j]]), acc);
        }
#pragma unroll
        for (int o = TPR >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (sub == 0 && row < n) y[row] = acc;
    }
}

static int pick_tpr(int32_t n, int64_t nnz) {
    const double mean = n > 0 ? (double)nnz / n : 1.0;
    if (mean <= 2.5) return 2;
    if (mean <= 6.0) return 4;
    if (mean <= 12.0) return 8;
    if (mean <= 24.0) return 16;
    return 32;
}

int csr_spmv_launch(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                    const int32_t* indices, const double* data, const double* x, double* y,
                    cudaStream_t st) {
    return csr_spmv_rows_launch(ctx, n, indptr, indices, data, x, y, n, nnz, st);
}

int csr_spmv_rows_launch(nodal_ctx* ctx, int32_t n, const int32_t* indptr, const int32_t* indices,
                         const double* data, const double* x, double* y, int32_t shape_n, int64_t shape_nnz,
                         cudaStream_t st) {
    if (n == 0) return NODAL_OK;
    const int tpr = pick_tpr(shape_n, shape_nnz);
    int64_t blocks = ((int64_t)n * tpr + SPMV_THREADS - 1) / SPMV_THREADS;
    const int64_t cap = (int64_t)ctx->num_sms * 8;
    const int grid = (int)(blocks < cap ? blocks : cap);
#define GO(T) csr_spmv_kernel<T><<<grid, SPMV_THREADS, 0, st>>>(n, indptr, indices, data, x, y)
    switch (tpr) {
        case 2: GO(2); break;
        case 4: GO(4); break;
        case 8: GO(8); break;
        case 16: GO(16); break;
        default: GO(32); break;
    }
#undef GO
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_spmv(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                          const int32_t* indices, const double* data, const double* x, double* y,
                          void* stream) {
    if (!ctx || n < 0) return NODAL_BAD_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    return csr_spmv_launch(ctx, n, nnz, indptr, indices, data, x, y, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- sliced ELL
// Census of the encoding (sell_core.cuh), one pass over the CSR entries next to the slice widths:
// flags[1] != 0 when an offset col - row does not fit int16; the nonzero value bit patterns go to a
// hash set per block, then to the global set gset, counted in flags[2].  +0.0 (the padding) is in
// every table and is the empty slot of the sets.  The counts stop growing soon after they pass the
// table size: a matrix with more distinct values is stored wide whatever the exact count.
constexpr int SELL_SET = 1024;   // slots of the hash sets (load factor <= 1/2 when counting stops)

__device__ __forceinline__ u32 sell_set_slot(u64 bits) {
    return (u32)((bits * 0x9E3779B97F4A7C15ull) >> 54);   // top 10 bits: SELL_SET slots
}

// Inserts bits != 0 into set: 1 when it was not there yet, 0 when it was, -1 when the set is full.
__device__ __forceinline__ int sell_set_insert(u64* set, u64 bits) {
    u32 h = sell_set_slot(bits);
    for (int probe = 0; probe < SELL_SET; ++probe, h = (h + 1) & (SELL_SET - 1)) {
        const u64 cur = set[h];
        if (cur == bits) return 0;
        if (cur == 0) {
            const u64 prev = atomicCAS(&set[h], 0ull, bits);
            if (prev == 0) return 1;
            if (prev == bits) return 0;
        }
    }
    return -1;
}

__global__ void __launch_bounds__(SPMV_THREADS)
sell_widths_kernel(int32_t n, int32_t nslices, const int32_t* __restrict__ indptr,
                   const int32_t* __restrict__ indices, const double* __restrict__ data,
                   const double* __restrict__ sc, int census, u32* __restrict__ slice_w,
                   u32* __restrict__ flags, u64* __restrict__ gset) {
    __shared__ u64 set[SELL_SET];
    __shared__ u32 count;
    if (census) {
        for (int i = threadIdx.x; i < SELL_SET; i += blockDim.x) set[i] = 0;
        if (threadIdx.x == 0) count = 0;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    bool far = false;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const int64_t r = s * 32 + lane;
        u32 len = 0;
        if (r < n) {
            const int32_t b = indptr[r], e = indptr[r + 1];
            len = (u32)(e - b);
            // values are read only while the matrix can still go compact as far as this thread knows
            for (int32_t j = b; census && j < e; ++j) {
                const int32_t c = indices[j];
                far |= !sell_offset_fits(c, r);
                if (far || *(volatile u32*)&count >= SELL_DICT_MAX) continue;
                double v = data[j];
                if (sc) v = (v * sc[r]) * sc[c];
                const u64 bits = sell_bits(v);
                if (bits != 0) {
                    const int added = sell_set_insert(set, bits);
                    if (added) atomicAdd(&count, added > 0 ? 1u : (u32)SELL_SET);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
        if (lane == 0) slice_w[s] = len;
    }
    if (!census) return;
    // a block that already knows the matrix stays wide does not merge its set
    if (__syncthreads_or(far)) {
        if (threadIdx.x == 0) flags[1] = 1;
        return;
    }
    if (count >= SELL_DICT_MAX) {
        if (threadIdx.x == 0) atomicAdd(&flags[2], (u32)SELL_SET);
        return;
    }
    for (int i = threadIdx.x; i < SELL_SET; i += blockDim.x) {
        const u64 bits = set[i];
        if (bits != 0 && *(volatile u32*)&flags[2] < SELL_DICT_MAX) {
            const int added = sell_set_insert(gset, bits);
            if (added) atomicAdd(&flags[2], added > 0 ? 1u : (u32)SELL_SET);   // full: more than the table holds
        }
    }
}

// dict[0] = +0.0, then the nonzero patterns of gset in increasing bit order; unused entries 0.
// One block of SELL_SET threads.
__global__ void __launch_bounds__(SELL_SET)
sell_dict_kernel(const u64* __restrict__ gset, u64* __restrict__ dict) {
    __shared__ u64 set[SELL_SET];
    __shared__ u64 out[SELL_DICT_MAX];
    const int t = threadIdx.x;
    set[t] = gset[t];
    if (t < SELL_DICT_MAX) out[t] = 0;
    __syncthreads();
    const u64 key = set[t];
    if (key != 0) {
        int rank = 1;
        for (int i = 0; i < SELL_SET; ++i) rank += set[i] != 0 && set[i] < key;
        out[rank] = key;
    }
    __syncthreads();
    if (t < SELL_DICT_MAX) dict[t] = out[t];
}

__global__ void __launch_bounds__(SPMV_THREADS)
sell_fill_kernel(int32_t n, int32_t nslices, const int32_t* __restrict__ indptr,
                 const int32_t* __restrict__ indices, const double* __restrict__ data,
                 const u32* __restrict__ slice_w, const double* __restrict__ sc,
                 int32_t* __restrict__ cols, double* __restrict__ vals,
                 const uint64_t* __restrict__ dict, int ndict, int16_t* __restrict__ dcol,
                 uint8_t* __restrict__ vidx, double* __restrict__ dinv) {
    __shared__ uint64_t sdict[SELL_DICT_MAX];
    const bool compact = dict != nullptr;
    if (compact) {
        for (int i = threadIdx.x; i < ndict; i += blockDim.x) sdict[i] = dict[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const int64_t r = s * 32 + lane;
        const u32 w0 = slice_w[s], w = slice_w[s + 1] - w0;
        int32_t b = 0, e = 0;
        if (r < n) { b = indptr[r]; e = indptr[r + 1]; }
        double diag = 0.0;
        const int64_t base = (int64_t)w0 * 32 + lane;
        for (u32 k = 0; k < w; ++k) {
            int32_t c = sell_pad_col(r, n);
            double v = 0.0;
            if (b + (int32_t)k < e) {
                c = indices[b + k];
                v = data[b + k];
                if (sc) v = (v * sc[r]) * sc[c];      // symmetric scaling: S A S
                if (c == r) diag += v;
            }
            const int64_t i = base + (int64_t)k * 32;
            if (compact) {
                dcol[i] = sell_encode_col(c, r);
                vidx[i] = sell_encode_val(sdict, ndict, sell_bits(v));
            } else {
                cols[i] = c;
                vals[i] = v;
            }
        }
        if (r < n) dinv[r] = diag != 0.0 ? 1.0 / diag : 1.0;
    }
}

void sell_free(nodal_sell* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    ctx_pool_free(m->ctx, m->slice_w);
    ctx_pool_free(m->ctx, m->store);
    ctx_pool_free(m->ctx, m->dinv);
    delete m;
}

int sell_from_csr(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                  const int32_t* indices, const double* data, nodal_sell** out, cudaStream_t st,
                  const double* sc) {
    *out = nullptr;
    nodal_sell* m = new nodal_sell();
    m->ctx = ctx;
    m->device = ctx->device;
    m->n = n;
    m->nnz = nnz;
    m->nslices = (n + 31) / 32;
    const int64_t ns = m->nslices;
    int rc = NODAL_OK;
    auto fail = [&](int code) { sell_free(m); return code; };
#define CT(expr)                                                                             \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            nodal_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                    \
                            cudaGetErrorString(_e));                                         \
            return fail(NODAL_CUDA_ERROR);                                                   \
        }                                                                                    \
    } while (0)
#define PA(field, type, bytes)                                                               \
    do {                                                                                     \
        m->field = static_cast<type*>(ctx_pool_alloc(ctx, (bytes)));                         \
        if (!m->field) {                                                                     \
            nodal_set_error("%s:%d: out of device memory (%zu bytes)", __FILE__, __LINE__,   \
                            (size_t)(bytes));                                                \
            return fail(NODAL_CUDA_ERROR);                                                   \
        }                                                                                    \
    } while (0)
    PA(slice_w, u32, sizeof(u32) * (size_t)(ns + 1));
    PA(dinv, double, sizeof(double) * (size_t)(n > 0 ? n : 1));
    CT(cudaMemsetAsync(m->slice_w, 0, sizeof(u32) * (size_t)(ns + 1), st));
    if (n == 0) { *out = m; return NODAL_OK; }
    const int census = getenv("NODAL_SELL_WIDE") ? 0 : 1;
    const int64_t cap = (int64_t)ctx->num_sms * 8;
    const int64_t want = (ns * 32 + SPMV_THREADS - 1) / SPMV_THREADS;
    const int grid = (int)(want < cap ? want : cap);
    rc = ctx_reserve(ctx, scan_scratch_bytes(ns + 1) + 4096 + sizeof(u64) * SELL_SET);
    if (rc != NODAL_OK) return fail(rc);
    u32* tot = carve<u32>(ctx, 16);     // [0] total width, [1] an offset does not fit, [2] distinct count
    u64* gset = carve<u64>(ctx, SELL_SET);
    CT(cudaMemsetAsync(tot, 0, sizeof(u32) * 16, st));
    CT(cudaMemsetAsync(gset, 0, sizeof(u64) * SELL_SET, st));
    sell_widths_kernel<<<grid, SPMV_THREADS, 0, st>>>(n, m->nslices, indptr, indices, data, sc, census,
                                                      m->slice_w, tot, gset);
    CT(cudaGetLastError());
    rc = scan_exclusive_u32(ctx, m->slice_w, m->slice_w, ns + 1, tot, st);
    if (rc != NODAL_OK) return fail(rc);
    u32* host_tot = reinterpret_cast<u32*>(ctx->pinned);
    CT(cudaMemcpyAsync(host_tot, tot, sizeof(u32) * 3, cudaMemcpyDeviceToHost, st));
    CT(cudaStreamSynchronize(st));
    m->padded = (int64_t)host_tot[0] * 32;
    m->compact = census && host_tot[1] == 0 && host_tot[2] + 1 <= (u32)SELL_DICT_MAX;   // + 1: the +0.0
    const size_t alloc = (size_t)(m->padded > 0 ? m->padded : 32);
    // one block so that a single L2 access-policy window can cover the operator
    if (m->compact) {
        m->ndict = (int32_t)host_tot[2] + 1;
        m->store_bytes = sizeof(double) * SELL_DICT_MAX + (sizeof(int16_t) + sizeof(uint8_t)) * alloc;
        PA(store, char, m->store_bytes);
        m->dict = static_cast<double*>(m->store);
        m->dcol = reinterpret_cast<int16_t*>(m->dict + SELL_DICT_MAX);
        m->vidx = reinterpret_cast<uint8_t*>(m->dcol + alloc);
        sell_dict_kernel<<<1, SELL_SET, 0, st>>>(gset, reinterpret_cast<u64*>(m->dict));
        CT(cudaGetLastError());
    } else {
        m->store_bytes = (sizeof(double) + sizeof(int32_t)) * alloc;
        PA(store, char, m->store_bytes);
        m->vals = static_cast<double*>(m->store);
        m->cols = reinterpret_cast<int32_t*>(m->vals + alloc);
    }
#undef PA
    sell_fill_kernel<<<grid, SPMV_THREADS, 0, st>>>(n, m->nslices, indptr, indices, data, m->slice_w, sc, m->cols,
                                                    m->vals, reinterpret_cast<const uint64_t*>(m->dict), m->ndict,
                                                    m->dcol, m->vidx, m->dinv);
    CT(cudaGetLastError());
#undef CT
    *out = m;
    return NODAL_OK;
}

// y = A x, one warp per slice, grid-stride over slices.
template <class A>
__global__ void __launch_bounds__(SPMV_THREADS, 5)
sell_spmv_kernel(int32_t n, int32_t nslices, const u32* __restrict__ slice_w, A a0,
                 const double* __restrict__ x, double* __restrict__ y) {
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int w = (int)(slice_w[s + 1] - w0);
        const int64_t base = (int64_t)w0 * 32 + lane;
        const int64_t r = s * 32 + lane;
        const double acc = sell_row_dot(a, base, r, w, x);
        if (r < n) y[r] = acc;
    }
}

extern "C" int nodal_sell_create(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                                 const int32_t* indices, const double* data, nodal_sell** out,
                                 void* stream) {
    if (!ctx || n < 0 || !out) return NODAL_BAD_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    return sell_from_csr(ctx, n, nnz, indptr, indices, data, out, (cudaStream_t)stream, nullptr);
}

extern "C" int nodal_sell_destroy(nodal_sell* m) {
    sell_free(m);
    return NODAL_OK;
}

extern "C" int64_t nodal_sell_padded_nnz(const nodal_sell* m) { return m ? m->padded : 0; }

extern "C" int nodal_sell_compact(const nodal_sell* m) { return m && m->compact ? 1 : 0; }

extern "C" int nodal_sell_spmv(nodal_ctx* ctx, const nodal_sell* m, const double* x, double* y,
                               void* stream) {
    if (!ctx || !m) return NODAL_BAD_ARG;
    if (m->n == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t want = ((int64_t)m->nslices * 32 + SPMV_THREADS - 1) / SPMV_THREADS;
    const int64_t cap = (int64_t)ctx->num_sms * 5;
    sell_launch(m, [&](auto a) {
        sell_spmv_kernel<<<(int)(want < cap ? want : cap), SPMV_THREADS, 0, (cudaStream_t)stream>>>(
            m->n, m->nslices, m->slice_w, a, x, y);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}
