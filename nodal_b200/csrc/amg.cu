// Aggregation AMG preconditioner + preconditioned CG in FP64 (opt-in alternative to the
// Jacobi-PCG of pcg.cu for the `spsolve(G, A)` call, nodal/nodal.py:325, on R / A netlists).
//
// Why: Jacobi-PCG needs O(sqrt(n)) iterations on grid-like networks (18 741 on the 4096 x 4096
// grid); a V-cycle over pairwise aggregates keeps the count nearly flat (31 .. 45 from 128^2 to
// 1024^2 in the numpy statement of this algorithm, tests/amg_mirror.py).
//
// Setup, per level (everything on the device, deterministic, no floating-point atomics):
//   * two passes of pairwise aggregation (Notay-style double pairwise): a handshake matching --
//     every unmatched row proposes to its preferred unmatched neighbour (amg_core.cuh), mutual
//     proposals become pairs, 8 rounds -- then rows left alone join the pair of their preferred
//     neighbour;
//   * aggregate ids = exclusive scan over the "I am the smallest index of my aggregate" flags;
//   * Galerkin operator P^T A P with piecewise-constant P: relabel every stored entry to
//     (agg[row], agg[col]) and hand the triples to the CSR builder the assembly path uses
//     (radix sort + in-order segmented sum, csr.cu), so coarse operators are bit-reproducible;
//   * P^T as a CSR pattern (same builder) so the restriction is a gather, not a scatter.
// Cycle: V(1,1) with damped Jacobi (omega), coarse correction scaled by `scale` (piecewise-
// constant prolongation under-corrects smooth error; 1.8 halves the iteration count), the
// coarsest operator (<= 512 rows by default) is inverted explicitly once (Gauss-Jordan) and
// applied as a dense mat-vec.  All operators are stored as SELL-32 (sparse.cuh).
#include <algorithm>
#include <cmath>

#include "amg_host.cuh"

void amg_free_csr(nodal_ctx* ctx, AmgCsr& a) {
    if (a.owned) {
        ctx_pool_free(ctx, const_cast<int32_t*>(a.indptr));
        ctx_pool_free(ctx, const_cast<int32_t*>(a.indices));
        ctx_pool_free(ctx, const_cast<double*>(a.data));
    }
    a = AmgCsr();
}

int amg_aggregate(nodal_ctx* ctx, int rounds, const AmgCsr& A, int32_t nown, int32_t base,
                  int32_t** agg_out, int32_t* nc_out, cudaStream_t st) {
    const int32_t n = A.n;
    AmgScratch<int32_t> match(ctx, n), best(ctx, n);
    AmgScratch<u32> leader(ctx, n);
    if (!match.ptr || !best.ptr || !leader.ptr) return NODAL_CUDA_ERROR;
    const int grid = amg_rows_grid(ctx, n);
    CUDA_TRY(cudaMemsetAsync(match, 0xFF, sizeof(int32_t) * (size_t)n, st));
    for (int r = 0; r < rounds; ++r) {
        amg_propose_kernel<<<grid, AT, 0, st>>>(n, A.indptr, A.indices, A.data, match, best, nown, base);
        KERNEL_CHECK();
        amg_accept_kernel<<<grid, AT, 0, st>>>(n, best, match);
        KERNEL_CHECK();
    }
    int32_t* root = best;       // the proposals are not needed any more
    amg_root_kernel<<<grid, AT, 0, st>>>(n, A.indptr, A.indices, A.data, match, root, leader, nown, base);
    KERNEL_CHECK();
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes(n) + 4096));
    u32* total = carve<u32>(ctx, 16);
    if (!total) return NODAL_CUDA_ERROR;
    NODAL_TRY(scan_exclusive_u32(ctx, leader, leader, n, total, st));
    int32_t* agg = match;       // nor is the matching
    amg_assign_kernel<<<grid, AT, 0, st>>>(n, root, leader, agg);
    KERNEL_CHECK();
    u32* total_h = reinterpret_cast<u32*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(total_h, total, sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *nc_out = (int32_t)total_h[0];
    *agg_out = match.keep();
    return NODAL_OK;
}

int amg_transpose_pattern(nodal_ctx* ctx, int32_t n, const int32_t* agg, int32_t** pt_ptr_out,
                          int32_t** pt_idx_out, cudaStream_t st) {
    AmgScratch<u64> keys(ctx, n);
    AmgScratch<double> vals(ctx, n), rhs(ctx, (size_t)n + 1), ones(ctx, n);
    if (!keys.ptr || !vals.ptr || !rhs.ptr || !ones.ptr) return NODAL_CUDA_ERROR;
    const int cb = amg_bit_length(n);
    amg_pt_keys_kernel<<<amg_rows_grid(ctx, n), AT, 0, st>>>(n, agg, cb, keys, vals);
    KERNEL_CHECK();
    int64_t cnt = 0;
    NODAL_TRY(nodal_csr_build(ctx, n, n, cb, reinterpret_cast<uint64_t*>(keys.ptr), vals, rhs, &cnt, st));
    if (cnt != n) {
        nodal_set_error("amg: internal error, P^T has %lld entries for %d rows", (long long)cnt, n);
        return NODAL_CUDA_ERROR;
    }
    AmgScratch<int32_t> pp(ctx, (size_t)n + 1), pi(ctx, n);
    if (!pp.ptr || !pi.ptr) return NODAL_CUDA_ERROR;
    NODAL_TRY(nodal_csr_fetch(ctx, n, n, pp, pi, ones, st));
    *pt_ptr_out = pp.keep();
    *pt_idx_out = pi.keep();
    return NODAL_OK;
}

int amg_members(nodal_ctx* ctx, int32_t n, const int32_t* agg, int32_t nc, int32_t** pt_ptr_out,
                int32_t** pt_idx_out, cudaStream_t st) {
    AmgScratch<u32> cnt(ctx, (size_t)nc + 1), cursor(ctx, (size_t)nc + 1);
    AmgScratch<int32_t> pp(ctx, (size_t)nc + 1), pi(ctx, (size_t)std::max(n, 1));
    if (!cnt.ptr || !cursor.ptr || !pp.ptr || !pi.ptr) return NODAL_CUDA_ERROR;
    CUDA_TRY(cudaMemsetAsync(cnt, 0, sizeof(u32) * ((size_t)nc + 1), st));
    CUDA_TRY(cudaMemsetAsync(cursor, 0, sizeof(u32) * ((size_t)nc + 1), st));
    const int grid = amg_rows_grid(ctx, n);
    amg_count_members_kernel<<<grid, AT, 0, st>>>(n, agg, cnt);
    KERNEL_CHECK();
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes((int64_t)nc + 1) + 4096));
    NODAL_TRY(scan_exclusive_u32(ctx, cnt, reinterpret_cast<u32*>(pp.ptr), (int64_t)nc + 1, nullptr, st));
    amg_place_members_kernel<<<grid, AT, 0, st>>>(n, agg, pp, cursor, pi);
    KERNEL_CHECK();
    amg_sort_members_kernel<<<amg_rows_grid(ctx, nc), AT, 0, st>>>(nc, pp, pi);
    KERNEL_CHECK();
    *pt_ptr_out = pp.keep();
    *pt_idx_out = pi.keep();
    return NODAL_OK;
}

int amg_galerkin_merge(nodal_ctx* ctx, const AmgCsr& A, const int32_t* pt_ptr, const int32_t* pt_idx, int32_t nc,
                       const int32_t* label, int32_t ncol_limit, AmgCsr* out, cudaStream_t st) {
    if (A.nnz >= ((int64_t)1 << 32) - 1) return NODAL_BAD_ARG;
    AmgScratch<u32> bound(ctx, (size_t)nc + 1), kept(ctx, (size_t)nc + 1);
    AmgScratch<int32_t> tmp_cols(ctx, (size_t)std::max<int64_t>(A.nnz, 1)), ip(ctx, (size_t)nc + 1);
    AmgScratch<double> tmp_vals(ctx, (size_t)std::max<int64_t>(A.nnz, 1));
    if (!bound.ptr || !kept.ptr || !tmp_cols.ptr || !tmp_vals.ptr || !ip.ptr) return NODAL_CUDA_ERROR;
    const int grid = amg_rows_grid(ctx, nc);
    CUDA_TRY(cudaMemsetAsync(bound.ptr + nc, 0, sizeof(u32), st));
    CUDA_TRY(cudaMemsetAsync(kept.ptr + nc, 0, sizeof(u32), st));
    amg_merge_bound_kernel<<<grid, AT, 0, st>>>(nc, pt_ptr, pt_idx, A.indptr, bound);
    KERNEL_CHECK();
    NODAL_TRY(ctx_reserve(ctx, scan_scratch_bytes((int64_t)nc + 1) + 4096));
    u32* total = carve<u32>(ctx, 16);
    if (!total) return NODAL_CUDA_ERROR;
    const size_t mark = ctx->arena_used;
    NODAL_TRY(scan_exclusive_u32(ctx, bound, bound, (int64_t)nc + 1, nullptr, st));
    ctx->arena_used = mark;
    amg_merge_rows_kernel<<<grid, AT, 0, st>>>(nc, pt_ptr, pt_idx, A.indptr, A.indices, A.data, label, ncol_limit,
                                               bound, tmp_cols, tmp_vals, kept);
    KERNEL_CHECK();
    NODAL_TRY(scan_exclusive_u32(ctx, kept, reinterpret_cast<u32*>(ip.ptr), (int64_t)nc + 1, total, st));
    u32* total_h = reinterpret_cast<u32*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(total_h, total, sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int64_t nnzc = total_h[0];
    AmgScratch<int32_t> ix(ctx, (size_t)std::max<int64_t>(nnzc, 1));
    AmgScratch<double> dv(ctx, (size_t)std::max<int64_t>(nnzc, 1));
    if (!ix.ptr || !dv.ptr) return NODAL_CUDA_ERROR;
    amg_merge_compact_kernel<<<grid, AT, 0, st>>>(nc, bound, ip, tmp_cols, tmp_vals, ix, dv);
    KERNEL_CHECK();
    out->n = nc;
    out->nnz = nnzc;
    out->indptr = ip.keep();
    out->indices = ix.keep();
    out->data = dv.keep();
    out->owned = true;
    return NODAL_OK;
}

namespace {

int rows_grid(const nodal_ctx* ctx, int64_t work) { return amg_rows_grid(ctx, work); }
int sell_grid(const nodal_ctx* ctx, int32_t nslices) { return amg_sell_grid(ctx, nslices); }
int bit_length(int64_t v) { return amg_bit_length(v); }
template <typename T>
T* pool(nodal_ctx* ctx, size_t count) { return amg_pool<T>(ctx, count); }
template <typename T>
using Scratch = AmgScratch<T>;
using Csr = AmgCsr;
void free_csr(nodal_ctx* ctx, Csr& a) { amg_free_csr(ctx, a); }
int aggregate(nodal_amg* h, const Csr& A, int32_t** agg_out, int32_t* nc_out, cudaStream_t st) {
    return amg_aggregate(h->ctx, h->rounds, A, 0x7fffffff, 0, agg_out, nc_out, st);
}

// Ac = P^T A P for the piecewise-constant P of `agg`.
bool sorted_galerkin() {
    static const bool on = getenv("NODAL_AMG_SORT_GALERKIN") != nullptr;
    return on;
}

int galerkin(nodal_amg* h, const Csr& A, const int32_t* agg, int32_t nc, Csr* out, cudaStream_t st) {
    nodal_ctx* ctx = h->ctx;
    if (!sorted_galerkin() && amg_merge_pays(A.nnz, nc)) {
        // sort-free: members of every aggregate, then one thread merges the member rows of its
        // coarse row (same summation order as the sort-based product below: bit-identical)
        int32_t *pp = nullptr, *pi = nullptr;
        NODAL_TRY(amg_members(ctx, A.n, agg, nc, &pp, &pi, st));
        const int rc = amg_galerkin_merge(ctx, A, pp, pi, nc, agg, 0x7fffffff, out, st);
        ctx_pool_free(ctx, pp);
        ctx_pool_free(ctx, pi);
        return rc;
    }
    Scratch<u64> keys(ctx, A.nnz);
    Scratch<double> vals(ctx, A.nnz), rhs(ctx, (size_t)nc + 1);
    if (!keys.ptr || !vals.ptr || !rhs.ptr) return NODAL_CUDA_ERROR;
    const int cb = bit_length(nc);
    amg_relabel_kernel<<<rows_grid(ctx, A.n), AT, 0, st>>>(A.n, A.indptr, A.indices, A.data, agg, cb,
                                                         keys, vals);
    KERNEL_CHECK();
    int64_t nnzc = 0;
    NODAL_TRY(nodal_csr_build(ctx, nc, A.nnz, cb, reinterpret_cast<uint64_t*>(keys.ptr), vals, rhs,
                              &nnzc, st));
    Scratch<int32_t> ip(ctx, (size_t)nc + 1), ix(ctx, nnzc);
    Scratch<double> dv(ctx, nnzc);
    if (!ip.ptr || !ix.ptr || !dv.ptr) return NODAL_CUDA_ERROR;
    NODAL_TRY(nodal_csr_fetch(ctx, nc, nnzc, ip, ix, dv, st));
    out->n = nc;
    out->nnz = nnzc;
    out->indptr = ip.keep();
    out->indices = ix.keep();
    out->data = dv.keep();
    out->owned = true;
    return NODAL_OK;
}

int transpose_pattern(nodal_amg* h, AmgLevel& L, cudaStream_t st) {
    if (!sorted_galerkin()) return amg_members(h->ctx, L.n, L.agg, L.nc, &L.pt_ptr, &L.pt_idx, st);
    return amg_transpose_pattern(h->ctx, L.n, L.agg, &L.pt_ptr, &L.pt_idx, st);
}

int invert_coarsest(nodal_amg* h, const AmgLevel& L, cudaStream_t st) {
    nodal_ctx* ctx = h->ctx;
    const int32_t n = L.n;
    const size_t elems = (size_t)n * 2 * n;
    Scratch<double> m0(ctx, elems + 32), m1(ctx, elems);
    if (!m0.ptr || !m1.ptr) return NODAL_CUDA_ERROR;
    int* bad = reinterpret_cast<int*>(m0.ptr + elems);
    CUDA_TRY(cudaMemsetAsync(m0, 0, sizeof(double) * (elems + 32), st));
    amg_dense_init_kernel<<<rows_grid(ctx, n), AT, 0, st>>>(n, L.indptr, L.indices, L.data, m0);
    KERNEL_CHECK();
    double *src = m0.ptr, *dst = m1.ptr;
    const int grid = rows_grid(ctx, (int64_t)elems);
    for (int32_t k = 0; k < n; ++k) {
        amg_gj_step_kernel<<<grid, AT, 0, st>>>(n, k, src, dst, bad);
        KERNEL_CHECK();
        std::swap(src, dst);
    }
    h->inv = pool<double>(ctx, (size_t)n * n);
    if (!h->inv) return NODAL_CUDA_ERROR;
    amg_dense_extract_kernel<<<rows_grid(ctx, (int64_t)n * n), AT, 0, st>>>(n, src, h->inv);
    KERNEL_CHECK();
    int* bad_h = reinterpret_cast<int*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(bad_h, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (*bad_h != 0) {
        nodal_set_error("amg: the coarsest operator is not positive definite (pivot %d of %d); "
                        "the matrix is not SPD", *bad_h, n);
        return NODAL_BREAKDOWN;
    }
    return NODAL_OK;
}

int build_hierarchy(nodal_amg* h, int32_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                    const double* data, cudaStream_t st) {
    nodal_ctx* ctx = h->ctx;
    Csr cur;
    cur.n = n; cur.nnz = nnz; cur.indptr = indptr; cur.indices = indices; cur.data = data;
    while (cur.n > h->coarse && (int)h->lv.size() < h->maxlevels) {
        Csr A = cur;            // borrowed view while A is the level operator itself
        A.owned = false;
        int32_t* comp = nullptr;
        int rc = NODAL_OK;
        for (int pass = 0; pass < h->passes && rc == NODAL_OK; ++pass) {
            int32_t* agg = nullptr;
            int32_t nc = 0;
            Csr Ac;
            rc = aggregate(h, A, &agg, &nc, st);
            if (rc == NODAL_OK) rc = galerkin(h, A, agg, nc, &Ac, st);
            if (rc == NODAL_OK && comp) {
                amg_compose_kernel<<<rows_grid(ctx, cur.n), AT, 0, st>>>(cur.n, comp, agg);
                ++g_nodal_launches;
                if (cudaGetLastError() != cudaSuccess) {
                    nodal_set_error("amg: amg_compose_kernel launch failed");
                    rc = NODAL_CUDA_ERROR;
                }
            }
            if (!comp) comp = agg;
            else ctx_pool_free(ctx, agg);
            free_csr(ctx, A);
            A = Ac;
        }
        // stalled: hardly fewer rows, or hardly fewer entries (expander-like graphs fill in: every
        // coarse row couples to the union of its members' neighbourhoods and the hierarchy would
        // cost more per level than it gains)
        // ... measured by the operator complexity the hierarchy would reach: sum of the levels'
        // entries over the finest level's)
        double total_nnz = (double)cur.nnz + (double)A.nnz;
        for (const AmgLevel& P : h->lv) total_nnz += (double)P.nnz;
        const bool too_dense = (double)A.nnz > h->max_fill * (double)cur.nnz ||
                               total_nnz > h->max_complexity * (double)(h->lv.empty() ? cur.nnz : h->lv[0].nnz);
        if (rc != NODAL_OK || (double)A.n > 0.9 * (double)cur.n || too_dense) {
            free_csr(ctx, A);       // error, or coarsening stalled: cur stays the coarsest level
            ctx_pool_free(ctx, comp);
            if (rc != NODAL_OK) {
                free_csr(ctx, cur);
                return rc;
            }
            break;
        }
        AmgLevel L;
        L.n = cur.n; L.nnz = cur.nnz; L.indptr = cur.indptr; L.indices = cur.indices; L.data = cur.data;
        L.owned = cur.owned;
        L.agg = comp;
        L.nc = A.n;
        h->lv.push_back(L);
        cur = A;
        rc = transpose_pattern(h, h->lv.back(), st);
        if (rc != NODAL_OK) {
            free_csr(ctx, cur);
            return rc;
        }
    }
    AmgLevel L;
    L.n = cur.n; L.nnz = cur.nnz; L.indptr = cur.indptr; L.indices = cur.indices; L.data = cur.data;
    L.owned = cur.owned;
    h->lv.push_back(L);
    for (size_t l = 0; l < h->lv.size(); ++l) {
        AmgLevel& V = h->lv[l];
        NODAL_TRY(sell_from_csr(ctx, V.n, V.nnz, V.indptr, V.indices, V.data, &V.sell, st, nullptr));
        V.x = pool<double>(ctx, V.n);
        V.r = pool<double>(ctx, V.n);
        if (l > 0) V.b = pool<double>(ctx, V.n);
        if (!V.x || !V.r || (l > 0 && !V.b)) return NODAL_CUDA_ERROR;
    }
    if (h->lv.back().n <= h->direct_max) NODAL_TRY(invert_coarsest(h, h->lv.back(), st));
    return NODAL_OK;
}

template <int MODE>
int sell_sweep(const nodal_amg* h, const AmgLevel& V, const double* b, const double* x, double* y,
               double* part, cudaStream_t st) {
    const nodal_sell* m = V.sell;
    sell_launch(m, [&](auto a) {
        amg_sell_kernel<MODE><<<sell_grid(h->ctx, m->nslices), AT, 0, st>>>(
            m->n, m->nslices, m->slice_w, a, m->dinv, b, x, h->omega, y, part);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}

// The fused sweeps of the cycle (amg_kernels.cuh): MODE 1 writes r = b - A x0 with x0 = omega D^-1 b,
// MODE 2 writes y = x~ + omega D^-1 (b - A x~) with x~ = x0 + scale P xc.
template <int MODE>
int cycle_sweep(const nodal_amg* h, const AmgLevel& V, const double* b, const double* xc, double* y,
                cudaStream_t st) {
    const nodal_sell* m = V.sell;
    sell_launch(m, [&](auto a) {
        amg_cycle_sweep_kernel<MODE><<<sell_grid(h->ctx, m->nslices), AT, 0, st>>>(
            m->n, m->nslices, m->slice_w, a, m->dinv, b, h->omega, V.agg, xc, h->scale, y);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}

// z = M b : one V(1,1) cycle from a zero initial guess.  Neither the Jacobi start x0 nor the
// prolongated iterate is stored: the sweeps form them where they gather (cycle_sweep).
int cycle(const nodal_amg* h, const double* b0, double* z0, cudaStream_t st) {
    const nodal_ctx* ctx = h->ctx;
    const int last = (int)h->lv.size() - 1;
    for (int l = 0; l < last; ++l) {
        const AmgLevel& V = h->lv[l];
        const double* b = l == 0 ? b0 : V.b;
        NODAL_TRY(cycle_sweep<1>(h, V, b, nullptr, V.r, st));
        amg_restrict_kernel<<<rows_grid(ctx, V.nc), AT, 0, st>>>(V.nc, V.pt_ptr, V.pt_idx, V.r,
                                                              h->lv[l + 1].b);
        KERNEL_CHECK();
    }
    {
        const AmgLevel& V = h->lv[last];
        const double* b = last == 0 ? b0 : V.b;
        double* x = last == 0 ? z0 : V.x;
        if (h->inv) amg_gemv_kernel<<<rows_grid(ctx, (int64_t)V.n * 32), AT, 0, st>>>(V.n, h->inv, b, x);
        else amg_jacobi0_kernel<<<rows_grid(ctx, V.n), AT, 0, st>>>(V.n, V.sell->dinv, b, h->omega, x);
        KERNEL_CHECK();
    }
    for (int l = last - 1; l >= 0; --l) {
        const AmgLevel& V = h->lv[l];
        const double* b = l == 0 ? b0 : V.b;
        NODAL_TRY(cycle_sweep<2>(h, V, b, h->lv[l + 1].x, l == 0 ? z0 : V.x, st));
    }
    return NODAL_OK;
}

}  // namespace

extern "C" int nodal_amg_destroy(nodal_amg* h) {
    if (!h) return NODAL_OK;
    cudaSetDevice(h->device);
    nodal_ctx* ctx = h->ctx;
    for (AmgLevel& V : h->lv) {
        sell_free(V.sell);
        if (V.owned) {
            ctx_pool_free(ctx, const_cast<int32_t*>(V.indptr));
            ctx_pool_free(ctx, const_cast<int32_t*>(V.indices));
            ctx_pool_free(ctx, const_cast<double*>(V.data));
        }
        ctx_pool_free(ctx, V.agg);
        ctx_pool_free(ctx, V.pt_ptr);
        ctx_pool_free(ctx, V.pt_idx);
        ctx_pool_free(ctx, V.b);
        ctx_pool_free(ctx, V.x);
        ctx_pool_free(ctx, V.r);
    }
    ctx_pool_free(ctx, h->inv);
    ctx_pool_free(ctx, h->p);
    ctx_pool_free(ctx, h->q);
    ctx_pool_free(ctx, h->r);
    ctx_pool_free(ctx, h->z);
    ctx_pool_free(ctx, h->part);
    delete h;
    return NODAL_OK;
}

extern "C" int nodal_amg_create(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                                const int32_t* indices, const double* data, const double* params,
                                nodal_amg** out, void* stream) {
    NvtxRange nvtx_range("nodal_amg_create");
    if (!ctx || n < 0 || nnz < 0 || !out) return NODAL_BAD_ARG;
    *out = nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    nodal_amg* h = new nodal_amg();
    h->ctx = ctx;
    h->device = ctx->device;
    if (params) {
        if (params[0] >= 1.0) h->passes = (int)params[0];
        if (params[1] >= 1.0) h->coarse = (int)params[1];
        if (params[2] > 0.0) h->omega = params[2];
        if (params[3] > 0.0) h->scale = params[3];
        if (params[4] >= 1.0) h->maxlevels = (int)params[4];
        if (params[5] >= 1.0) h->rounds = (int)params[5];
        if (params[6] >= 1.0) h->direct_max = (int)params[6];
        if (params[7] > 0.0) h->max_fill = params[7];
    }
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    cudaEventRecord(e0, st);
    int rc = NODAL_OK;
    if (n > 0) rc = build_hierarchy(h, n, nnz, indptr, indices, data, st);
    if (rc == NODAL_OK && n > 0) {
        h->nparts = std::max(sell_grid(ctx, h->lv[0].sell->nslices), rows_grid(ctx, n));
        h->p = pool<double>(ctx, n);
        h->q = pool<double>(ctx, n);
        h->r = pool<double>(ctx, n);
        h->z = pool<double>(ctx, n);
        h->part = pool<double>(ctx, 3 * (size_t)h->nparts + 16);
        if (!h->p || !h->q || !h->r || !h->z || !h->part) rc = NODAL_CUDA_ERROR;
    }
    cudaEventRecord(e1, st);
    if (cudaEventSynchronize(e1) == cudaSuccess) cudaEventElapsedTime(&h->setup_ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc != NODAL_OK) {
        nodal_amg_destroy(h);
        return rc;
    }
    *out = h;
    return NODAL_OK;
}

extern "C" int nodal_amg_info(const nodal_amg* h, int32_t cap, int32_t* nlevels, int64_t* rows,
                              int64_t* nnz, double* setup_ms, int32_t* direct) {
    if (!h || !nlevels) return NODAL_BAD_ARG;
    *nlevels = (int32_t)h->lv.size();
    for (int32_t l = 0; l < *nlevels && l < cap; ++l) {
        if (rows) rows[l] = h->lv[l].n;
        if (nnz) nnz[l] = h->lv[l].nnz;
    }
    if (setup_ms) *setup_ms = h->setup_ms;
    if (direct) *direct = h->inv ? 1 : 0;
    return NODAL_OK;
}

extern "C" int nodal_amg_fetch_level(nodal_ctx* ctx, const nodal_amg* h, int32_t level, int32_t* agg,
                                     int32_t* indptr, int32_t* indices, double* data, void* stream) {
    if (!ctx || !h || level < 0 || level >= (int32_t)h->lv.size()) return NODAL_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const AmgLevel& V = h->lv[level];
    if (agg) {
        if (!V.agg) return NODAL_BAD_ARG;   // the coarsest level has no aggregates
        CUDA_TRY(cudaMemcpyAsync(agg, V.agg, sizeof(int32_t) * (size_t)V.n, cudaMemcpyDeviceToDevice, st));
    }
    if (indptr) CUDA_TRY(cudaMemcpyAsync(indptr, V.indptr, sizeof(int32_t) * ((size_t)V.n + 1), cudaMemcpyDeviceToDevice, st));
    if (indices) CUDA_TRY(cudaMemcpyAsync(indices, V.indices, sizeof(int32_t) * (size_t)V.nnz, cudaMemcpyDeviceToDevice, st));
    if (data) CUDA_TRY(cudaMemcpyAsync(data, V.data, sizeof(double) * (size_t)V.nnz, cudaMemcpyDeviceToDevice, st));
    return NODAL_OK;
}

extern "C" int nodal_amg_apply(nodal_ctx* ctx, const nodal_amg* h, const double* r, double* z,
                               void* stream) {
    if (!ctx || !h || h->ctx != ctx) return NODAL_BAD_ARG;
    if (h->lv.empty()) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    return cycle(h, r, z, (cudaStream_t)stream);
}

extern "C" int nodal_amg_pcg(nodal_ctx* ctx, nodal_amg* h, const double* rhs, double* x, double rtol,
                             int32_t maxit, int32_t* iters_h, double* relres_h, double* stats_h,
                             void* stream) {
    NvtxRange nvtx_range("nodal_amg_pcg");
    if (!ctx || !h || h->ctx != ctx || !iters_h || !relres_h) return NODAL_BAD_ARG;
    *iters_h = 0;
    *relres_h = 0.0;
    if (stats_h) memset(stats_h, 0, 16 * sizeof(double));
    if (h->lv.empty()) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const AmgLevel& A = h->lv[0];
    const int32_t n = A.n;
    const int gv = rows_grid(ctx, n);                        // vector kernels
    const int gs = sell_grid(ctx, A.sell->nslices);          // SELL sweeps
    double* part_pq = h->part;
    double* part_rr = h->part + h->nparts;
    double* part_rz = h->part + 2 * (size_t)h->nparts;
    double* scal = h->part + 3 * (size_t)h->nparts;          // [0..1] rz (parity), [2] norm scratch
    double* host = reinterpret_cast<double*>(ctx->pinned);
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    int iters = 0, restarts = 0, rc = NODAL_NOT_CONVERGED;
    double relres = 0.0;
    bool timed = false;

    // ||v||^2 of a device vector pair -> host
    auto dot_to_host = [&](const double* a, const double* b, double* result) -> int {
        apcg_dot_kernel<<<gv, AT, 0, st>>>(n, a, b, part_rr);
        KERNEL_CHECK();
        apcg_sum_kernel<<<1, AT, 0, st>>>(part_rr, gv, scal + 2);
        KERNEL_CHECK();
        CUDA_TRY(cudaMemcpyAsync(host, scal + 2, sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        *result = host[0];
        return NODAL_OK;
    };
    auto run = [&]() -> int {
        CUDA_TRY(cudaEventRecord(e0, st));
        double bb = 0.0, rr = 0.0;
        NODAL_TRY(dot_to_host(rhs, rhs, &bb));
        if (!(bb > 0.0)) {                                   // b = 0 -> x = 0
            if (bb == 0.0) {
                CUDA_TRY(cudaMemsetAsync(x, 0, sizeof(double) * (size_t)n, st));
                rc = NODAL_OK;
                return NODAL_OK;
            }
            nodal_set_error("nodal_amg_pcg: the right-hand side is not finite");
            rc = NODAL_BREAKDOWN;
            return NODAL_OK;
        }
        const double bnorm = sqrt(bb);
        NODAL_TRY(sell_sweep<1>(h, A, rhs, x, h->r, nullptr, st));       // r = b - A x0
        NODAL_TRY(dot_to_host(h->r, h->r, &rr));
        relres = sqrt(rr) / bnorm;
        while (true) {
            if (relres <= rtol) { rc = NODAL_OK; break; }
            if (iters >= maxit) { rc = NODAL_NOT_CONVERGED; break; }
            if (restarts > 8) { rc = NODAL_NOT_CONVERGED; break; }
            // (re)start from the current r
            int par = 0;
            NODAL_TRY(cycle(h, h->r, h->z, st));
            apcg_dot_kernel<<<gv, AT, 0, st>>>(n, h->r, h->z, part_rz);
            KERNEL_CHECK();
            apcg_direction_kernel<<<gv, AT, 0, st>>>(n, part_rz, gv, scal + (par ^ 1), scal + par, h->z, h->p, 1);
            KERNEL_CHECK();
            bool broke = false;
            while (iters < maxit) {
                NODAL_TRY(sell_sweep<0>(h, A, nullptr, h->p, h->q, part_pq, st));
                apcg_update_kernel<<<gv, AT, 0, st>>>(n, part_pq, gs, scal + par, h->p, h->q, x, h->r, part_rr);
                KERNEL_CHECK();
                apcg_sum_kernel<<<1, AT, 0, st>>>(part_rr, gv, scal + 2);
                KERNEL_CHECK();
                CUDA_TRY(cudaMemcpyAsync(host, scal + 2, sizeof(double), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                ++iters;
                rr = host[0];
                if (!std::isfinite(rr)) { broke = true; break; }
                if (sqrt(rr) <= rtol * bnorm) break;
                NODAL_TRY(cycle(h, h->r, h->z, st));
                apcg_dot_kernel<<<gv, AT, 0, st>>>(n, h->r, h->z, part_rz);
                KERNEL_CHECK();
                apcg_direction_kernel<<<gv, AT, 0, st>>>(n, part_rz, gv, scal + par, scal + (par ^ 1), h->z, h->p, 0);
                KERNEL_CHECK();
                par ^= 1;
            }
            if (broke) {
                nodal_set_error("nodal_amg_pcg: breakdown (non-finite residual) at iteration %d", iters);
                rc = NODAL_BREAKDOWN;
                break;
            }
            // the recurrence says converged (or maxit): check the true residual
            NODAL_TRY(sell_sweep<1>(h, A, rhs, x, h->r, nullptr, st));
            NODAL_TRY(dot_to_host(h->r, h->r, &rr));
            relres = sqrt(rr) / bnorm;
            if (!std::isfinite(relres)) { rc = NODAL_BREAKDOWN; break; }
            if (relres > rtol) ++restarts;
        }
        CUDA_TRY(cudaEventRecord(e1, st));
        CUDA_TRY(cudaEventSynchronize(e1));
        timed = true;
        return NODAL_OK;
    };
    const int st_run = run();
    float ms = 0.f;
    if (st_run == NODAL_OK && timed) cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (st_run != NODAL_OK) return st_run;
    *iters_h = iters;
    *relres_h = relres;
    if (stats_h) {
        double rows = 0.0, nnz = 0.0;
        for (const AmgLevel& V : h->lv) { rows += V.n; nnz += (double)V.nnz; }
        stats_h[0] = (double)h->lv.size();
        stats_h[1] = A.nnz ? nnz / (double)A.nnz : 0.0;       // operator complexity
        stats_h[2] = restarts;
        stats_h[3] = ms;
        stats_h[4] = h->setup_ms;
        stats_h[5] = h->lv.back().n;
        stats_h[6] = n ? rows / n : 0.0;                       // grid complexity
        stats_h[7] = h->inv ? 1.0 : 0.0;
    }
    return rc;
}

// Per-launch time of the level-0 SELL sweeps (the dominant kernels of the AMG-PCG step) for the
// roofline entry of bench.py: `reps` launches of each mode on the hierarchy's own level-0
// operator and work vectors, bracketed by CUDA events on `stream`.
// ms_out[0] = MODE 0 (q = A p + dot), [1] = MODE 1 (residual), [2] = MODE 2 (Jacobi sweep).
extern "C" int nodal_amg_profile_sweeps(nodal_ctx* ctx, nodal_amg* h, int32_t reps, double* ms_out, void* stream) {
    if (!ctx || !h || h->ctx != ctx || !ms_out || reps < 1 || h->lv.empty()) return NODAL_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const AmgLevel& A = h->lv[0];
    CUDA_TRY(cudaMemsetAsync(h->p, 0, sizeof(double) * (size_t)A.n, st));
    CUDA_TRY(cudaMemsetAsync(h->r, 0, sizeof(double) * (size_t)A.n, st));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    int rc = NODAL_OK;
    for (int mode = 0; mode < 3 && rc == NODAL_OK; ++mode) {
        for (int k = -2; k < reps && rc == NODAL_OK; ++k) {      // two warm-up launches
            if (k == 0) cudaEventRecord(e0, st);
            if (mode == 0) rc = sell_sweep<0>(h, A, nullptr, h->p, h->q, h->part, st);
            if (mode == 1) rc = sell_sweep<1>(h, A, h->r, h->p, h->q, nullptr, st);
            if (mode == 2) rc = sell_sweep<2>(h, A, h->r, h->p, h->q, nullptr, st);
        }
        cudaEventRecord(e1, st);
        float ms = 0.f;
        if (cudaEventSynchronize(e1) == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
        ms_out[mode] = ms / reps;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return rc;
}

// Per-launch time of the level-0 kernels of the V-cycle, unfused and fused, for
// benchmarks/amg_cycle.py: `reps` launches each (after two warm-up launches) on the hierarchy's own
// level-0 operator, aggregates and work vectors, bracketed by CUDA events on `stream`.
// ms_out: [0] jacobi0, [1] MODE 1 residual, [2] prolong, [3] MODE 2 Jacobi sweep,
//         [4] fused residual of the Jacobi start, [5] fused post-smoothing.
extern "C" int nodal_amg_profile_cycle(nodal_ctx* ctx, nodal_amg* h, int32_t reps, double* ms_out, void* stream) {
    if (!ctx || !h || h->ctx != ctx || !ms_out || reps < 1 || h->lv.size() < 2) return NODAL_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const AmgLevel& A = h->lv[0];
    const AmgLevel& C = h->lv[1];
    double* b = h->r;
    CUDA_TRY(cudaMemsetAsync(b, 0, sizeof(double) * (size_t)A.n, st));
    CUDA_TRY(cudaMemsetAsync(A.x, 0, sizeof(double) * (size_t)A.n, st));
    CUDA_TRY(cudaMemsetAsync(C.x, 0, sizeof(double) * (size_t)C.n, st));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    int rc = NODAL_OK;
    for (int k = 0; k < 6 && rc == NODAL_OK; ++k) {
        for (int i = -2; i < reps && rc == NODAL_OK; ++i) {
            if (i == 0) cudaEventRecord(e0, st);
            switch (k) {
                case 0:
                    amg_jacobi0_kernel<<<rows_grid(ctx, A.n), AT, 0, st>>>(A.n, A.sell->dinv, b, h->omega, A.x);
                    KERNEL_CHECK();
                    break;
                case 1: rc = sell_sweep<1>(h, A, b, A.x, A.r, nullptr, st); break;
                case 2:
                    amg_prolong_kernel<<<rows_grid(ctx, A.n), AT, 0, st>>>(A.n, A.agg, C.x, h->scale, A.x, A.r);
                    KERNEL_CHECK();
                    break;
                case 3: rc = sell_sweep<2>(h, A, b, A.r, h->z, nullptr, st); break;
                case 4: rc = cycle_sweep<1>(h, A, b, nullptr, A.r, st); break;
                default: rc = cycle_sweep<2>(h, A, b, C.x, h->z, st); break;
            }
        }
        cudaEventRecord(e1, st);
        float ms = 0.f;
        if (cudaEventSynchronize(e1) == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
        ms_out[k] = ms / reps;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return rc;
}
