// Shared declarations for libnodal_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/nodal_b200.h"

#include <nvtx3/nvToolsExt.h>

// NVTX range over a scope (header-only NVTX v3: a no-op unless a profiler is attached), so nsys /
// ncu timelines show the stages of the path by name (SURVEY.md section 5).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

typedef unsigned long long u64;
typedef unsigned int u32;

#define NODAL_NUM_SMS_FALLBACK 148

void nodal_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            nodal_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                \
                            cudaGetErrorString(_e));                                     \
            (void)cudaGetLastError(); /* clear non-sticky errors */                      \
            return NODAL_CUDA_ERROR;                                                     \
        }                                                                                \
    } while (0)

#define NODAL_TRY(expr)                                                                  \
    do {                                                                                 \
        int _s = (expr);                                                                 \
        if (_s != NODAL_OK) return _s;                                                   \
    } while (0)

extern unsigned long long g_nodal_launches;  // kernels launched by this library (host counter)
#define KERNEL_CHECK()                 \
    do {                               \
        ++g_nodal_launches;            \
        CUDA_TRY(cudaGetLastError());  \
    } while (0)

// A grow-only device scratch arena.  Each API call opens a Scope, carves what it
// needs and everything is handed back when the Scope dies.  If the arena is too
// small it is re-allocated (after a device sync) -- only outside hot loops.
struct nodal_ctx {
    int device = 0;
    int num_sms = NODAL_NUM_SMS_FALLBACK;
    char* arena = nullptr;
    size_t arena_bytes = 0;
    size_t arena_used = 0;
    uint64_t generation = 0;  // bumped by every ctx_reserve (invalidates pending results)
    // pinned host scratch for status words
    void* pinned = nullptr;
    // cache of long-lived device buffers (solver-private matrix copies, halo tables ...):
    // cudaMalloc / cudaFree cost milliseconds when several processes share a node
    struct PoolBlock { void* ptr; size_t bytes; bool used; };
    std::vector<PoolBlock> pool;
};

void* ctx_pool_alloc(nodal_ctx* ctx, size_t bytes);   // nullptr on failure
void ctx_pool_free(nodal_ctx* ctx, void* ptr);

int ctx_reserve(nodal_ctx* ctx, size_t bytes);  // make sure arena holds >= bytes (resets it)
void* ctx_carve(nodal_ctx* ctx, size_t bytes);  // 256-B aligned bump allocation (nullptr if full)

template <typename T>
static inline T* carve(nodal_ctx* ctx, size_t count) {
    return reinterpret_cast<T*>(ctx_carve(ctx, count * sizeof(T)));
}
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lanemask_lt() {
    u32 m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Block-wide sum for blocks of up to 1024 threads; result valid in every thread.
// Fixed shuffle tree -> deterministic.
__device__ __forceinline__ double block_sum(double v, double* smem /* >= 33 doubles */) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane_id() == 0) smem[w] = v;
    __syncthreads();
    if (w == 0) {
        double t = (lane_id() < nw) ? smem[lane_id()] : 0.0;
        t = warp_sum(t);
        if (lane_id() == 0) smem[32] = t;
    }
    __syncthreads();
    return smem[32];
}

// Deterministic sum of `count` partials (written by a previous kernel) computed
// redundantly by every block: fixed assignment of partials to threads + fixed tree.
__device__ __forceinline__ double reduce_partials(const double* __restrict__ part, int count,
                                                  double* smem) {
    double t = 0.0;
    for (int i = threadIdx.x; i < count; i += blockDim.x) t += part[i];
    return block_sum(t, smem);
}

// The same for up to three arrays at once with every load in flight before the first add
// (three dependent-latency loops cost ~5 us at the head of a 90 us kernel).  Each thread adds
// its values in the same order as reduce_partials, so the results are bit-identical.
// Counts must be <= 8 * blockDim.x; pass count 0 / nullptr for unused slots.
__device__ __forceinline__ void reduce_partials3(const double* __restrict__ a, int na,
                                                 const double* __restrict__ b, int nb,
                                                 const double* __restrict__ c, int nc, double* smem,
                                                 double& sa, double& sb, double& sc) {
    double va[8], vb[8], vc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = threadIdx.x + k * blockDim.x;
        va[k] = i < na ? a[i] : 0.0;
        vb[k] = i < nb ? b[i] : 0.0;
        vc[k] = i < nc ? c[i] : 0.0;
    }
    double ta = 0.0, tb = 0.0, tc = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = threadIdx.x + k * blockDim.x;
        if (i < na) ta += va[k];
        if (i < nb) tb += vb[k];
        if (i < nc) tc += vc[k];
    }
    sa = block_sum(ta, smem);
    sb = nb > 0 ? block_sum(tb, smem) : 0.0;
    sc = nc > 0 ? block_sum(tc, smem) : 0.0;
}
#endif

// kernels implemented in other translation units
int scan_exclusive_u32(nodal_ctx* ctx, const u32* in, u32* out, int64_t count, u32* total_dev,
                       cudaStream_t st);
size_t scan_scratch_bytes(int64_t count);
int radix_sort_pairs(nodal_ctx* ctx, u64* keys, u64* vals, u64* keys_alt, u64* vals_alt,
                     int64_t count, int bits, bool* result_in_alt, cudaStream_t st);
size_t radix_sort_scratch_bytes(int64_t count);
int radix_sort_check(nodal_ctx* ctx);
int cc_union_find(nodal_ctx* ctx, int64_t nedges, const int32_t* rows, const int32_t* a, const int32_t* b,
                  int32_t kcl, int32_t* parent, int32_t* labels, cudaStream_t st);   // csrc/graph.cu   // after a stream sync: NODAL_CUDA_ERROR if a sort pass gave up
