// Elimination of independent voltage sources (E rows) from an R / A / E netlist, so that the
// SPD solvers (AMG-PCG) handle it: the reference's spsolve of the indefinite MNA system
// (nodal/nodal.py:325) is replaced by a solve of the reduced weighted Laplacian plus an exact
// expansion.  The per-item rules are in sources_core.cuh; tests/sources_mirror.py states the
// whole algorithm in numpy.
//
//   nodal_source_forest        E rows -> forest over the nodes: union-find (csrc/graph.cu) counts the
//                              loops; when there are none, every tree is oriented from its root by a
//                              level-synchronous BFS (one launch per level) giving rep_row, offset,
//                              parent_edge and depth per node; roots not in ground's tree are
//                              numbered in row order (the reduced rows).
//   nodal_source_reduce_scan / nodal_source_reduce_table
//                              ordered flag / scan / place of the component table into the reduced
//                              R / A table (component order kept).
//   nodal_source_expand        potentials from the reduced solution, KCL residual with the full G,
//                              subtree sums level by level from the deepest, source currents, and
//                              the relative residual of the full system.
//   nodal_source_potentials / _tree_rows / _currents / _residual
//                              the same expansion in stages for a rank of the row-partitioned solve
//                              (nodal_b200/dist_sources.py), launching the same kernels.
//
// Nothing accumulates floating-point values with atomics: results are bitwise reproducible.
#include <algorithm>

#include "sources_core.cuh"
#include "sparse.cuh"

constexpr int ST = 256;

static int src_grid(nodal_ctx* ctx, int64_t work) {
    int64_t g = (work + ST - 1) / ST;
    const int64_t cap = (int64_t)ctx->num_sms * 16;
    return (int)(g < 1 ? 1 : g < cap ? g : cap);
}

#define GRID_STRIDE(i, count) \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (count); i += (int64_t)gridDim.x * blockDim.x)

// ---------------------------------------------------------------- forest
__global__ void __launch_bounds__(ST)
src_flag_e_kernel(int64_t ncomp, const uint8_t* __restrict__ type, u32* __restrict__ flag) {
    GRID_STRIDE(i, ncomp) flag[i] = type[i] == NODAL_T_E ? 1u : 0u;
}

__global__ void __launch_bounds__(ST)
src_place_e_kernel(int64_t ncomp, const uint8_t* __restrict__ type, const u32* __restrict__ pos, int32_t cap,
                   int32_t* __restrict__ erow) {
    GRID_STRIDE(i, ncomp) {
        if (type[i] == NODAL_T_E && pos[i] < (u32)cap) erow[pos[i]] = (int32_t)i;
    }
}

// integer atomics only: per-branch use counts, per-node source degrees
__global__ void __launch_bounds__(ST)
src_degree_kernel(int32_t nsrc, const int32_t* __restrict__ erow, const int32_t* __restrict__ a,
                  const int32_t* __restrict__ b, const int32_t* __restrict__ branch, int32_t kcl, int32_t be,
                  u32* __restrict__ deg, u32* __restrict__ used) {
    GRID_STRIDE(k, nsrc) {
        const int32_t r = erow[k];
        atomicAdd(&deg[src_node(a[r], kcl)], 1u);
        atomicAdd(&deg[src_node(b[r], kcl)], 1u);
        const int32_t br = branch[r];
        if (br >= 0 && br < be) atomicAdd(&used[br], 1u);
    }
}

// counts: [0] touched nodes, [1] trees, [2] branches not used exactly once, [3] nodes in ground's tree,
// [4] trees without ground (a tree's label is its smallest node, so it is counted at that node)
__global__ void __launch_bounds__(ST)
src_count_kernel(int32_t kcl, int32_t be, const u32* __restrict__ deg, const u32* __restrict__ used,
                 const int32_t* __restrict__ labels, u32* __restrict__ counts) {
    const int32_t glabel = labels[kcl];
    u32 c[5] = {0, 0, 0, 0, 0};
    GRID_STRIDE(v, (int64_t)kcl + 1) {
        const bool t = deg[v] > 0, head = t && labels[v] == (int32_t)v;
        c[0] += t;
        c[1] += head;
        c[3] += t && v < kcl && labels[v] == glabel;
        c[4] += head && labels[v] != glabel;
    }
    GRID_STRIDE(k, be) c[2] += used[k] != 1u;
#pragma unroll
    for (int q = 0; q < 5; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c[q] += __shfl_xor_sync(0xffffffffu, c[q], o);
        if ((threadIdx.x & 31) == 0 && c[q]) atomicAdd(&counts[q], c[q]);   // integer sums: order-free
    }
}

// half-edges of the adjacency: key = node << 32 | other node (sorted: per node, children in index order)
__global__ void __launch_bounds__(ST)
src_halfedge_kernel(int32_t nsrc, const int32_t* __restrict__ erow, const int32_t* __restrict__ a,
                    const int32_t* __restrict__ b, int32_t kcl, u64* __restrict__ keys, u64* __restrict__ vals) {
    GRID_STRIDE(k, nsrc) {
        const int32_t r = erow[k];
        const u64 u = (u64)src_node(a[r], kcl), w = (u64)src_node(b[r], kcl);
        keys[2 * k] = u << 32 | w;
        vals[2 * k] = (u64)r;
        keys[2 * k + 1] = w << 32 | u;
        vals[2 * k + 1] = (u64)r;
    }
}

__global__ void __launch_bounds__(ST)
src_adj_kernel(int64_t nhalf, const u64* __restrict__ vals, int32_t* __restrict__ adj_row) {
    GRID_STRIDE(j, nhalf) adj_row[j] = (int32_t)vals[j];
}

// root of a node: ground (kcl) for ground's tree, else the smallest node of the tree (its label)
__device__ __forceinline__ int32_t src_root(const int32_t* labels, int32_t v, int32_t kcl) {
    const int32_t l = labels[v];
    return l == labels[kcl] ? kcl : l;
}

__global__ void __launch_bounds__(ST)
src_free_root_kernel(int32_t kcl, const int32_t* __restrict__ labels, u32* __restrict__ flag) {
    GRID_STRIDE(v, (int64_t)kcl + 1) flag[v] = (v < kcl && src_root(labels, (int32_t)v, kcl) == (int32_t)v) ? 1u : 0u;
}

__global__ void __launch_bounds__(ST)
src_init_nodes_kernel(int32_t kcl, const int32_t* __restrict__ labels, const u32* __restrict__ red,
                      int32_t* __restrict__ rep_row, double* __restrict__ offset, int32_t* __restrict__ parent_edge,
                      int32_t* __restrict__ depth, int32_t* __restrict__ roots) {
    GRID_STRIDE(v, (int64_t)kcl + 1) {
        const int32_t r = src_root(labels, (int32_t)v, kcl);
        rep_row[v] = r == kcl ? NODAL_GROUND : (int32_t)red[r];
        offset[v] = 0.0;
        parent_edge[v] = -1;
        depth[v] = r == (int32_t)v ? 0 : -1;
        if (v < kcl && r == (int32_t)v) roots[red[v]] = (int32_t)v;
    }
}

// one BFS level: a node at depth `level` claims its unvisited neighbours.  In a forest every node
// has exactly one neighbour one level up, so every write below has a single writer.
__global__ void __launch_bounds__(ST)
src_bfs_level_kernel(int64_t nhalf, const u64* __restrict__ keys, const int32_t* __restrict__ adj_row,
                     const double* __restrict__ value, const int32_t* __restrict__ a, int32_t kcl, int32_t level,
                     int32_t* __restrict__ depth, double* __restrict__ offset, int32_t* __restrict__ parent_edge,
                     int32_t* __restrict__ changed) {
    GRID_STRIDE(j, nhalf) {
        const u64 key = keys[j];
        const int32_t u = (int32_t)(key >> 32), w = (int32_t)(key & 0xffffffffu);
        if (depth[u] != level || depth[w] >= 0) continue;
        const int32_t r = adj_row[j];
        depth[w] = level + 1;
        parent_edge[w] = r;
        offset[w] = src_child_offset(offset[u], value[r], src_node(a[r], kcl) == w);
        *changed = 1;
    }
}

extern "C" int nodal_source_forest(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const double* value,
                                   const int32_t* a, const int32_t* b, const int32_t* branch, int32_t kcl,
                                   int32_t be, int32_t* erow, int32_t* adj_ptr, int32_t* adj_row, int32_t* rep_row,
                                   double* offset, int32_t* parent_edge, int32_t* depth, int32_t* roots,
                                   int64_t* info_h, void* stream) {
    if (!ctx || ncomp < 0 || kcl < 0 || be < 0 || !info_h || ncomp >= ((int64_t)1 << 32) ||
        2 * (int64_t)be >= ((int64_t)1 << 30))
        return NODAL_BAD_ARG;
    NvtxRange nvtx_range("nodal_source_forest");
    cudaStream_t st = (cudaStream_t)stream;
    for (int k = 0; k < 8; ++k) info_h[k] = 0;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t nodes = kcl + 1;
    const int64_t nhalf = 2 * (int64_t)be;
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes(ncomp) + scan_scratch_bytes((int64_t)nodes + 1) +
                                   radix_sort_scratch_bytes(std::max<int64_t>(nhalf, 2)) + 65536));
    u32* dcount = carve<u32>(ctx, 16);
    int32_t* changed = reinterpret_cast<int32_t*>(dcount + 8);
    if (!dcount) return NODAL_CUDA_ERROR;
    void* bufs[8] = {};
    size_t sizes[8] = {sizeof(u32) * (size_t)std::max<int64_t>(ncomp, (int64_t)nodes + 1),   // flags / scans
                       sizeof(int32_t) * (size_t)nodes,                                   // union-find parent
                       sizeof(int32_t) * (size_t)nodes,                                   // labels
                       sizeof(u32) * ((size_t)nodes + 1),                                 // degrees
                       sizeof(u32) * (size_t)std::max(be, 1),                             // branch use
                       sizeof(u64) * (size_t)std::max<int64_t>(nhalf, 1),                 // keys
                       sizeof(u64) * (size_t)std::max<int64_t>(nhalf, 1)};                // vals
    auto release = [&]() {
        for (void* p : bufs) ctx_pool_free(ctx, p);
    };
    auto run = [&]() -> int {
        // the alternate sort buffers: the keys of the BFS must survive the sort, so two more
        sizes[7] = 2 * sizes[5];
        for (int k = 0; k < 8; ++k) {
            bufs[k] = ctx_pool_alloc(ctx, sizes[k]);
            if (!bufs[k]) {
                nodal_set_error("nodal_source_forest: out of device memory");
                return NODAL_CUDA_ERROR;
            }
        }
        u32* flag = static_cast<u32*>(bufs[0]);
        int32_t* parent = static_cast<int32_t*>(bufs[1]);
        int32_t* labels = static_cast<int32_t*>(bufs[2]);
        u32* deg = static_cast<u32*>(bufs[3]);
        u32* used = static_cast<u32*>(bufs[4]);
        u64* keys = static_cast<u64*>(bufs[5]);
        u64* vals = static_cast<u64*>(bufs[6]);
        u64* keys_alt = static_cast<u64*>(bufs[7]);
        u64* vals_alt = keys_alt + std::max<int64_t>(nhalf, 1);
        u32* host = reinterpret_cast<u32*>(ctx->pinned);

        // 1. the E rows in table order
        CUDA_TRY(cudaMemsetAsync(dcount, 0, 16 * sizeof(u32), st));
        if (ncomp > 0) {
            src_flag_e_kernel<<<src_grid(ctx, ncomp), ST, 0, st>>>(ncomp, type, flag);
            KERNEL_CHECK();
            NODAL_TRY(scan_exclusive_u32(ctx, flag, flag, ncomp, dcount, st));
            src_place_e_kernel<<<src_grid(ctx, ncomp), ST, 0, st>>>(ncomp, type, flag, be, erow);
            KERNEL_CHECK();
        }
        CUDA_TRY(cudaMemcpyAsync(host, dcount, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        const int64_t nE = host[0];
        info_h[0] = nE;
        if (nE != be) {              // some branch is not owned by exactly one E row
            info_h[2] = nE > be ? nE - be : be - nE;
            return NODAL_OK;
        }
        const int32_t nsrc = (int32_t)nE;

        // 2. union-find over the source edges, degrees, branch use
        NODAL_TRY(cc_union_find(ctx, nsrc, erow, a, b, kcl, parent, labels, st));
        CUDA_TRY(cudaMemsetAsync(deg, 0, sizeof(u32) * ((size_t)nodes + 1), st));
        CUDA_TRY(cudaMemsetAsync(used, 0, sizeof(u32) * (size_t)std::max(be, 1), st));
        CUDA_TRY(cudaMemsetAsync(dcount, 0, 8 * sizeof(u32), st));   // counters, numbering total
        if (nsrc > 0) {
            src_degree_kernel<<<src_grid(ctx, nsrc), ST, 0, st>>>(nsrc, erow, a, b, branch, kcl, be, deg, used);
            KERNEL_CHECK();
        }
        src_count_kernel<<<src_grid(ctx, std::max<int64_t>(nodes, be)), ST, 0, st>>>(kcl, be, deg, used, labels,
                                                                                     dcount);
        KERNEL_CHECK();
        CUDA_TRY(cudaMemcpyAsync(host, dcount, 5 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        const int64_t touched = host[0], trees = host[1];
        info_h[1] = nE - (touched - trees);     // independent loops of the source graph (self-loops included)
        info_h[2] = host[2];
        info_h[3] = trees;
        info_h[4] = host[4];
        info_h[5] = host[3];
        if (info_h[1] != 0 || info_h[2] != 0) return NODAL_OK;

        // 3. adjacency: per node its incident sources, ordered by the other node
        NODAL_TRY(scan_exclusive_u32(ctx, deg, reinterpret_cast<u32*>(adj_ptr), (int64_t)nodes + 1, nullptr, st));
        bool in_alt = false;
        if (nsrc > 0) {
            src_halfedge_kernel<<<src_grid(ctx, nsrc), ST, 0, st>>>(nsrc, erow, a, b, kcl, keys, vals);
            KERNEL_CHECK();
            int bits = 32;
            while (bits < 64 && ((u64)kcl >> (bits - 32)) != 0) ++bits;
            NODAL_TRY(radix_sort_pairs(ctx, keys, vals, keys_alt, vals_alt, nhalf, bits, &in_alt, st));
            if (in_alt) {
                std::swap(keys, keys_alt);
                std::swap(vals, vals_alt);
            }
            src_adj_kernel<<<src_grid(ctx, nhalf), ST, 0, st>>>(nhalf, vals, adj_row);
            KERNEL_CHECK();
        }

        // 4. roots, numbering of the reduced rows, BFS from the roots
        src_free_root_kernel<<<src_grid(ctx, nodes), ST, 0, st>>>(kcl, labels, flag);
        KERNEL_CHECK();
        NODAL_TRY(scan_exclusive_u32(ctx, flag, flag, nodes, dcount + 5, st));
        src_init_nodes_kernel<<<src_grid(ctx, nodes), ST, 0, st>>>(kcl, labels, flag, rep_row, offset, parent_edge,
                                                                   depth, roots);
        KERNEL_CHECK();
        int32_t* changed_h = reinterpret_cast<int32_t*>(host + 8);
        CUDA_TRY(cudaMemcpyAsync(host + 5, dcount + 5, sizeof(u32), cudaMemcpyDeviceToHost, st));
        int32_t level = 0;
        while (nsrc > 0) {
            CUDA_TRY(cudaMemsetAsync(changed, 0, sizeof(int32_t), st));
            src_bfs_level_kernel<<<src_grid(ctx, nhalf), ST, 0, st>>>(nhalf, keys, adj_row, value, a, kcl, level,
                                                                      depth, offset, parent_edge, changed);
            KERNEL_CHECK();
            CUDA_TRY(cudaMemcpyAsync(changed_h, changed, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (!*changed_h) break;
            ++level;
        }
        CUDA_TRY(cudaStreamSynchronize(st));
        NODAL_TRY(radix_sort_check(ctx));
        info_h[6] = host[5];
        info_h[7] = level;
        return NODAL_OK;
    };
    const int rc = run();
    release();
    return rc;
}

// ---------------------------------------------------------------- table reduction
__global__ void __launch_bounds__(ST)
src_reduce_flag_kernel(int64_t ncomp, const uint8_t* __restrict__ type, const int32_t* __restrict__ a,
                       const int32_t* __restrict__ b, int32_t kcl, const int32_t* __restrict__ rep_row,
                       const double* __restrict__ offset, u32* __restrict__ pos) {
    GRID_STRIDE(i, ncomp) pos[i] = (u32)src_reduce_count(type[i], a[i], b[i], kcl, rep_row, offset);
}

__global__ void __launch_bounds__(ST)
src_reduce_place_kernel(int64_t ncomp, const uint8_t* __restrict__ type, const double* __restrict__ value,
                        const int32_t* __restrict__ a, const int32_t* __restrict__ b, int32_t kcl,
                        const int32_t* __restrict__ rep_row, const double* __restrict__ offset,
                        const u32* __restrict__ pos, uint8_t* __restrict__ o_type, double* __restrict__ o_value,
                        int32_t* __restrict__ o_a, int32_t* __restrict__ o_b) {
    GRID_STRIDE(i, ncomp) {
        ReducedRows o;
        src_reduce_component(type[i], value[i], a[i], b[i], kcl, rep_row, offset, o);
        const u32 p = pos[i];
        for (int k = 0; k < o.count; ++k) {
            o_type[p + k] = o.type[k];
            o_value[p + k] = o.value[k];
            o_a[p + k] = o.a[k];
            o_b[p + k] = o.b[k];
        }
    }
}

extern "C" int nodal_source_reduce_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                                        const int32_t* b, int32_t kcl, const int32_t* rep_row, const double* offset,
                                        uint32_t* pos, int64_t* count_h, void* stream) {
    if (!ctx || ncomp < 0 || !count_h || ncomp >= ((int64_t)1 << 31)) return NODAL_BAD_ARG;
    *count_h = 0;
    if (ncomp == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes(ncomp) + 4096));
    u32* total = carve<u32>(ctx, 16);
    if (!total) return NODAL_CUDA_ERROR;
    src_reduce_flag_kernel<<<src_grid(ctx, ncomp), ST, 0, st>>>(ncomp, type, a, b, kcl, rep_row, offset, pos);
    KERNEL_CHECK();
    NODAL_TRY(scan_exclusive_u32(ctx, pos, pos, ncomp, total, st));
    u32* total_h = reinterpret_cast<u32*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(total_h, total, sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *count_h = total_h[0];
    return NODAL_OK;
}

extern "C" int nodal_source_reduce_table(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const double* value,
                                         const int32_t* a, const int32_t* b, int32_t kcl, const int32_t* rep_row,
                                         const double* offset, const uint32_t* pos, uint8_t* out_type,
                                         double* out_value, int32_t* out_a, int32_t* out_b, void* stream) {
    if (!ctx || ncomp < 0) return NODAL_BAD_ARG;
    if (ncomp == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    src_reduce_place_kernel<<<src_grid(ctx, ncomp), ST, 0, st>>>(ncomp, type, value, a, b, kcl, rep_row, offset, pos,
                                                                 out_type, out_value, out_a, out_b);
    KERNEL_CHECK();
    return NODAL_OK;
}

// ---------------------------------------------------------------- expansion
__global__ void __launch_bounds__(ST)
src_potentials_kernel(int32_t kcl, int32_t n, const int32_t* __restrict__ rep_row, const double* __restrict__ offset,
                      const double* __restrict__ y, double* __restrict__ x) {
    GRID_STRIDE(v, n) x[v] = v < kcl ? src_potential(rep_row[v], offset[v], y) : 0.0;
}

// Sources whose child sits at depth `level`: acc[c] = (rhs - Gx)[c] + the children's sums in the order of
// the adjacency (by node index); `gx` holds G x on entry and the subtree sums of the deeper levels.
__global__ void __launch_bounds__(ST)
src_subtree_level_kernel(int32_t nsrc, const int32_t* __restrict__ erow, const int32_t* __restrict__ a,
                         const int32_t* __restrict__ b, const int32_t* __restrict__ branch, int32_t kcl,
                         const int32_t* __restrict__ adj_ptr, const int32_t* __restrict__ adj_row,
                         const int32_t* __restrict__ depth, int32_t level, const double* __restrict__ rhs,
                         double* __restrict__ gx, double* __restrict__ x) {
    GRID_STRIDE(k, nsrc) {
        const int32_t r = erow[k];
        const int32_t u = src_node(a[r], kcl), w = src_node(b[r], kcl);
        const int32_t c = depth[u] > depth[w] ? u : w;
        if (depth[c] != level) continue;
        double s = rhs[c] - gx[c];
        for (int32_t j = adj_ptr[c]; j < adj_ptr[c + 1]; ++j) {
            const int32_t r2 = adj_row[j];
            const int32_t p = src_node(a[r2], kcl), q = src_node(b[r2], kcl);
            const int32_t o = p == c ? q : p;
            if (depth[o] == level + 1) s += gx[o];
        }
        gx[c] = s;
        x[kcl + branch[r]] = src_current(s, c == u);
    }
}

// per-block partial sums of (rhs - Gx)^2 and rhs^2, then one block adds the partials in a fixed order
__global__ void __launch_bounds__(ST)
src_residual_partials_kernel(int32_t n, const double* __restrict__ rhs, const double* __restrict__ gx,
                             double* __restrict__ part) {
    __shared__ double smem[33];
    double rr = 0.0, bb = 0.0;
    GRID_STRIDE(i, n) {
        const double r = rhs[i] - gx[i];
        rr += r * r;
        bb += rhs[i] * rhs[i];
    }
    rr = block_sum(rr, smem);
    bb = block_sum(bb, smem);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = rr;
        part[gridDim.x + blockIdx.x] = bb;
    }
}

__global__ void __launch_bounds__(ST)
src_residual_final_kernel(int nparts, const double* __restrict__ part, double* __restrict__ out) {
    __shared__ double smem[33];
    const double rr = reduce_partials(part, nparts, smem);
    const double bb = reduce_partials(part + nparts, nparts, smem);
    if (threadIdx.x == 0) {
        out[0] = rr;
        out[1] = bb;
    }
}

extern "C" int nodal_source_expand(nodal_ctx* ctx, int32_t kcl, int32_t n, int32_t nsrc, const int32_t* erow,
                                   const int32_t* a, const int32_t* b, const int32_t* branch, const int32_t* adj_ptr,
                                   const int32_t* adj_row, const int32_t* rep_row, const double* offset,
                                   const int32_t* depth, int32_t max_depth, const double* y, const double* rhs,
                                   int64_t nnz, const int32_t* indptr, const int32_t* indices, const double* data,
                                   double* x, double* relres_h, void* stream) {
    if (!ctx || kcl < 0 || n < kcl || nsrc < 0 || max_depth < 0 || !relres_h) return NODAL_BAD_ARG;
    NvtxRange nvtx_range("nodal_source_expand");
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int parts = src_grid(ctx, n);
    double* gx = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (size_t)std::max(n, 1)));
    double* part = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (2 * (size_t)parts + 2)));
    auto run = [&]() -> int {
        if (!gx || !part) {
            nodal_set_error("nodal_source_expand: out of device memory");
            return NODAL_CUDA_ERROR;
        }
        src_potentials_kernel<<<parts, ST, 0, st>>>(kcl, n, rep_row, offset, y, x);
        KERNEL_CHECK();
        NODAL_TRY(csr_spmv_launch(ctx, n, nnz, indptr, indices, data, x, gx, st));
        for (int32_t level = max_depth; level >= 1 && nsrc > 0; --level) {
            src_subtree_level_kernel<<<src_grid(ctx, nsrc), ST, 0, st>>>(nsrc, erow, a, b, branch, kcl, adj_ptr,
                                                                         adj_row, depth, level, rhs, gx, x);
            KERNEL_CHECK();
        }
        NODAL_TRY(csr_spmv_launch(ctx, n, nnz, indptr, indices, data, x, gx, st));
        src_residual_partials_kernel<<<parts, ST, 0, st>>>(n, rhs, gx, part);
        KERNEL_CHECK();
        src_residual_final_kernel<<<1, ST, 0, st>>>(parts, part, part + 2 * parts);
        KERNEL_CHECK();
        double* host = reinterpret_cast<double*>(ctx->pinned);
        CUDA_TRY(cudaMemcpyAsync(host, part + 2 * parts, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        *relres_h = host[1] > 0.0 ? sqrt(host[0] / host[1]) : sqrt(host[0]);
        return NODAL_OK;
    };
    const int rc = run();
    ctx_pool_free(ctx, gx);
    ctx_pool_free(ctx, part);
    return rc;
}

// ---------------------------------------------------------------- expansion in stages (row-partitioned)
// The stages of nodal_source_expand for a rank that holds rows [rb, re) of the full MNA matrix
// (row pointer rebased to 0, global columns) and the replicated forest of the E-only table.  They
// launch the kernels above; the row products take their lanes per row from the whole matrix's
// shape, so every rank forms G x on its rows exactly as the single-GPU expansion does.
__global__ void __launch_bounds__(ST)
src_tree_flag_kernel(int32_t rows, int32_t rb, int32_t kcl, const int32_t* __restrict__ depth, u32* __restrict__ flag) {
    GRID_STRIDE(i, rows) {
        const int64_t v = rb + i;
        flag[i] = (v < kcl && depth[v] >= 1) ? 1u : 0u;
    }
}

__global__ void __launch_bounds__(ST)
src_tree_place_kernel(int32_t rows, int32_t rb, int32_t kcl, const int32_t* __restrict__ depth,
                      const u32* __restrict__ pos, const double* __restrict__ rhs, const double* __restrict__ gx,
                      int32_t* __restrict__ o_row, double* __restrict__ o_rhs, double* __restrict__ o_gx) {
    GRID_STRIDE(i, rows) {
        const int64_t v = rb + i;
        if (!(v < kcl && depth[v] >= 1)) continue;
        const u32 p = pos[i];
        o_row[p] = (int32_t)v;
        o_rhs[p] = rhs[i];
        o_gx[p] = gx[i];
    }
}

__global__ void __launch_bounds__(ST)
src_tree_scatter_kernel(int32_t count, const int32_t* __restrict__ row, const double* __restrict__ t_rhs,
                        const double* __restrict__ t_gx, double* __restrict__ rhs, double* __restrict__ gx) {
    GRID_STRIDE(k, count) {
        rhs[row[k]] = t_rhs[k];
        gx[row[k]] = t_gx[k];
    }
}

extern "C" int nodal_source_potentials(nodal_ctx* ctx, int32_t kcl, int32_t n, const int32_t* rep_row,
                                       const double* offset, const double* y, double* x, void* stream) {
    if (!ctx || kcl < 0 || n < kcl) return NODAL_BAD_ARG;
    if (n == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    src_potentials_kernel<<<src_grid(ctx, n), ST, 0, (cudaStream_t)stream>>>(kcl, n, rep_row, offset, y, x);
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_source_tree_rows(nodal_ctx* ctx, int32_t kcl, int32_t n, int64_t nnz_full, int32_t rb, int32_t re,
                                      const int32_t* depth, const double* rhs, int64_t nnz, const int32_t* indptr,
                                      const int32_t* indices, const double* data, const double* x, int32_t* out_row,
                                      double* out_rhs, double* out_gx, int64_t* count_h, void* stream) {
    if (!ctx || kcl < 0 || n < kcl || rb < 0 || re < rb || re > n || nnz < 0 || !count_h) return NODAL_BAD_ARG;
    *count_h = 0;
    const int32_t rows = re - rb;
    if (rows == 0) return NODAL_OK;
    NvtxRange nvtx_range("nodal_source_tree_rows");
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes(rows) + 4096));
    u32* total = carve<u32>(ctx, 16);
    if (!total) return NODAL_CUDA_ERROR;
    double* gx = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (size_t)rows));
    u32* pos = static_cast<u32*>(ctx_pool_alloc(ctx, sizeof(u32) * (size_t)rows));
    auto run = [&]() -> int {
        if (!gx || !pos) {
            nodal_set_error("nodal_source_tree_rows: out of device memory");
            return NODAL_CUDA_ERROR;
        }
        NODAL_TRY(csr_spmv_rows_launch(ctx, rows, indptr, indices, data, x, gx, n, nnz_full, st));
        src_tree_flag_kernel<<<src_grid(ctx, rows), ST, 0, st>>>(rows, rb, kcl, depth, pos);
        KERNEL_CHECK();
        NODAL_TRY(scan_exclusive_u32(ctx, pos, pos, rows, total, st));
        src_tree_place_kernel<<<src_grid(ctx, rows), ST, 0, st>>>(rows, rb, kcl, depth, pos, rhs, gx, out_row, out_rhs,
                                                                  out_gx);
        KERNEL_CHECK();
        u32* total_h = reinterpret_cast<u32*>(ctx->pinned);
        CUDA_TRY(cudaMemcpyAsync(total_h, total, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        *count_h = total_h[0];
        return NODAL_OK;
    };
    const int rc = run();
    ctx_pool_free(ctx, gx);
    ctx_pool_free(ctx, pos);
    return rc;
}

extern "C" int nodal_source_currents(nodal_ctx* ctx, int32_t kcl, int32_t nsrc, const int32_t* erow, const int32_t* a,
                                     const int32_t* b, const int32_t* branch, const int32_t* adj_ptr,
                                     const int32_t* adj_row, const int32_t* depth, int32_t max_depth, int64_t ntree,
                                     const int32_t* tree_row, const double* tree_rhs, const double* tree_gx, double* x,
                                     void* stream) {
    if (!ctx || kcl < 0 || nsrc < 0 || max_depth < 0 || ntree < 0 || ntree > kcl) return NODAL_BAD_ARG;
    if (nsrc == 0 || max_depth == 0) return NODAL_OK;
    NvtxRange nvtx_range("nodal_source_currents");
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    // node-indexed rhs and G x; only the nodes at depth >= 1 (the tree rows) are read
    double* rhs = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * ((size_t)kcl + 1)));
    double* gx = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * ((size_t)kcl + 1)));
    auto run = [&]() -> int {
        if (!rhs || !gx) {
            nodal_set_error("nodal_source_currents: out of device memory");
            return NODAL_CUDA_ERROR;
        }
        if (ntree > 0) {
            src_tree_scatter_kernel<<<src_grid(ctx, ntree), ST, 0, st>>>((int32_t)ntree, tree_row, tree_rhs, tree_gx,
                                                                         rhs, gx);
            KERNEL_CHECK();
        }
        for (int32_t level = max_depth; level >= 1; --level) {
            src_subtree_level_kernel<<<src_grid(ctx, nsrc), ST, 0, st>>>(nsrc, erow, a, b, branch, kcl, adj_ptr,
                                                                         adj_row, depth, level, rhs, gx, x);
            KERNEL_CHECK();
        }
        return NODAL_OK;
    };
    const int rc = run();
    ctx_pool_free(ctx, rhs);
    ctx_pool_free(ctx, gx);
    return rc;
}

extern "C" int nodal_source_residual(nodal_ctx* ctx, int32_t n, int64_t nnz_full, int32_t rows, const double* rhs,
                                     int64_t nnz, const int32_t* indptr, const int32_t* indices, const double* data,
                                     const double* x, double* sums_h, void* stream) {
    if (!ctx || rows < 0 || rows > n || nnz < 0 || !sums_h) return NODAL_BAD_ARG;
    sums_h[0] = sums_h[1] = 0.0;
    if (rows == 0) return NODAL_OK;
    NvtxRange nvtx_range("nodal_source_residual");
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int parts = src_grid(ctx, rows);
    double* gx = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (size_t)rows));
    double* part = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (2 * (size_t)parts + 2)));
    auto run = [&]() -> int {
        if (!gx || !part) {
            nodal_set_error("nodal_source_residual: out of device memory");
            return NODAL_CUDA_ERROR;
        }
        NODAL_TRY(csr_spmv_rows_launch(ctx, rows, indptr, indices, data, x, gx, n, nnz_full, st));
        src_residual_partials_kernel<<<parts, ST, 0, st>>>(rows, rhs, gx, part);
        KERNEL_CHECK();
        src_residual_final_kernel<<<1, ST, 0, st>>>(parts, part, part + 2 * parts);
        KERNEL_CHECK();
        double* host = reinterpret_cast<double*>(ctx->pinned);
        CUDA_TRY(cudaMemcpyAsync(host, part + 2 * parts, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        sums_h[0] = host[0];
        sums_h[1] = host[1];
        return NODAL_OK;
    };
    const int rc = run();
    ctx_pool_free(ctx, gx);
    ctx_pool_free(ctx, part);
    return rc;
}
