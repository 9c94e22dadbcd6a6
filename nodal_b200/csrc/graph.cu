// Connectivity of the lead graph on the device: replaces the reference's breadth-first search
// `is_connected` (nodal/nodal.py:88-105, O(V^2) list membership tests, only reachable from the
// dense error path) for the diagnosis of singular systems (SURVEY.md section 8(f) rank 3).
//
// Nodes are the kcl rows plus ground (index kcl); every component contributes the edge
// anode - bnode (control nodes do not connect anything, as in the reference).  Lock-free
// union-find: one pass over the components hooks the larger root under the smaller one with a
// compare-and-swap (retrying when another thread got there first), `find` halves the path with
// plain stores to non-root entries, then every node is pointed at its root.  Parents only ever
// decrease, so there are no cycles; the result (the smallest index of each component as its
// label) does not depend on the schedule.
#include "common.cuh"

constexpr int GT = 256;

// Loads are volatile: other CTAs change `parent` while we walk it and L1 is not coherent -- a
// stale "I am a root" line would make the compare-and-swap below fail forever.
__device__ __forceinline__ int32_t cc_find(int32_t* parent, int32_t u) {
    volatile int32_t* vp = parent;
    while (true) {
        const int32_t p = vp[u];
        if (p == u) return u;
        const int32_t gp = vp[p];
        if (gp != p) vp[u] = gp;   // path halving; u is not a root, roots change only by CAS
        u = p;
    }
}

__global__ void __launch_bounds__(GT)
cc_init_kernel(int32_t nodes, int32_t* __restrict__ parent) {
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nodes;
         v += (int64_t)gridDim.x * blockDim.x)
        parent[v] = (int32_t)v;
}

__global__ void __launch_bounds__(GT)
cc_hook_kernel(int64_t ncomp, const int32_t* __restrict__ rows, const int32_t* __restrict__ a,
               const int32_t* __restrict__ b, int32_t kcl, int32_t* parent) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncomp;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = rows ? rows[i] : i;
        int32_t u = a[e], v = b[e];
        if (u < 0) u = kcl;              // ground lead
        if (v < 0) v = kcl;
        if (u > kcl || v > kcl) continue;   // validated on the host; never index out of range
        while (true) {
            u = cc_find(parent, u);
            v = cc_find(parent, v);
            if (u == v) break;
            const int32_t hi = u > v ? u : v, lo = u > v ? v : u;
            const int32_t seen = atomicCAS(&parent[hi], hi, lo);
            if (seen == hi) break;      // hooked
            u = seen;                   // somebody else hooked `hi` first: continue from its new parent
            v = lo;
        }
    }
}

// labels[v] = root of v; counts[0] += number of roots, counts[1] += nodes whose root is ground's
__global__ void __launch_bounds__(GT)
cc_label_kernel(int32_t nodes, int32_t* parent, int32_t* __restrict__ labels) {
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nodes;
         v += (int64_t)gridDim.x * blockDim.x)
        labels[v] = cc_find(parent, (int32_t)v);
}

__global__ void __launch_bounds__(GT)
cc_count_kernel(int32_t nodes, const int32_t* __restrict__ labels, int32_t* __restrict__ counts) {
    const int32_t ground_label = labels[nodes - 1];
    int roots = 0, reached = 0;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nodes;
         v += (int64_t)gridDim.x * blockDim.x) {
        const int32_t l = labels[v];
        roots += l == (int32_t)v;
        reached += l == ground_label;
    }
    // integer sums: the order of the atomics does not change the result
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        roots += __shfl_xor_sync(0xffffffffu, roots, o);
        reached += __shfl_xor_sync(0xffffffffu, reached, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (roots) atomicAdd(&counts[0], roots);
        if (reached) atomicAdd(&counts[1], reached);
    }
}

static int cc_grid(nodal_ctx* ctx, int64_t work) {
    int64_t g = (work + GT - 1) / GT;
    const int64_t cap = (int64_t)ctx->num_sms * 16;
    return (int)(g < 1 ? 1 : g < cap ? g : cap);
}

// labels[v] = smallest node of v's component over the edges a[e] - b[e], e = rows[i] for i < nedges
// (rows == nullptr: e = i).  `parent` is scratch of kcl + 1 entries.  Shared with csrc/sources.cu.
int cc_union_find(nodal_ctx* ctx, int64_t nedges, const int32_t* rows, const int32_t* a, const int32_t* b,
                  int32_t kcl, int32_t* parent, int32_t* labels, cudaStream_t st) {
    const int32_t nodes = kcl + 1;
    cc_init_kernel<<<cc_grid(ctx, nodes), GT, 0, st>>>(nodes, parent);
    KERNEL_CHECK();
    if (nedges > 0) {
        cc_hook_kernel<<<cc_grid(ctx, nedges), GT, 0, st>>>(nedges, rows, a, b, kcl, parent);
        KERNEL_CHECK();
    }
    cc_label_kernel<<<cc_grid(ctx, nodes), GT, 0, st>>>(nodes, parent, labels);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_connected_components(nodal_ctx* ctx, int64_t ncomp, const int32_t* a,
                                          const int32_t* b, int32_t kcl, int32_t* labels,
                                          int32_t* ncomponents_h, int32_t* reached_h, void* stream) {
    if (!ctx || ncomp < 0 || kcl < 0 || !ncomponents_h || !reached_h) return NODAL_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t nodes = kcl + 1;
    int32_t* parent = static_cast<int32_t*>(ctx_pool_alloc(ctx, sizeof(int32_t) * (size_t)nodes));
    int32_t* own_labels = nullptr;
    if (!labels) {
        own_labels = static_cast<int32_t*>(ctx_pool_alloc(ctx, sizeof(int32_t) * (size_t)nodes));
        labels = own_labels;
    }
    int32_t* counts = static_cast<int32_t*>(ctx_pool_alloc(ctx, 256));
    auto release = [&]() {
        ctx_pool_free(ctx, parent);
        ctx_pool_free(ctx, own_labels);
        ctx_pool_free(ctx, counts);
    };
    if (!parent || !labels || !counts) {
        release();
        nodal_set_error("nodal_connected_components: out of device memory");
        return NODAL_CUDA_ERROR;
    }
    auto run = [&]() -> int {
        CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
        NODAL_TRY(cc_union_find(ctx, ncomp, nullptr, a, b, kcl, parent, labels, st));
        cc_count_kernel<<<cc_grid(ctx, nodes), GT, 0, st>>>(nodes, labels, counts);
        KERNEL_CHECK();
        int32_t* host = reinterpret_cast<int32_t*>(ctx->pinned);
        CUDA_TRY(cudaMemcpyAsync(host, counts, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        *ncomponents_h = host[0];
        *reached_h = host[1];
        return NODAL_OK;
    };
    const int rc = run();
    release();
    return rc;
}
