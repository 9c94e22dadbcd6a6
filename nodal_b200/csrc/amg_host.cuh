// Host-side building blocks of the AMG setup shared by amg.cu (single GPU) and dist_amg.cu
// (row-partitioned): pool-backed scratch buffers, launch grids, one pairwise aggregation pass
// and the transposed prolongation pattern.
#pragma once
#include "amg_kernels.cuh"

static inline int amg_rows_grid(const nodal_ctx* ctx, int64_t work) {
    int64_t b = (work + AT - 1) / AT;
    const int64_t cap = (int64_t)ctx->num_sms * 16;
    if (b < 1) b = 1;
    return (int)(b < cap ? b : cap);
}
static inline int amg_sell_grid(const nodal_ctx* ctx, int32_t nslices) {
    int64_t b = ((int64_t)nslices * 32 + AT - 1) / AT;
    const int64_t cap = (int64_t)ctx->num_sms * 5;    // 5 CTAs / SM: what took the PCG's SELL kernel from 0.88 to 0.98 of peak
    if (b < 1) b = 1;
    return (int)(b < cap ? b : cap);
}
static inline int amg_bit_length(int64_t v) {
    int b = 1;
    while ((v >> b) != 0) ++b;
    return b;
}

template <typename T>
static inline T* amg_pool(nodal_ctx* ctx, size_t count) {
    T* p = static_cast<T*>(ctx_pool_alloc(ctx, sizeof(T) * (count ? count : 1)));
    if (!p) nodal_set_error("amg: out of device memory (%zu bytes)", sizeof(T) * count);
    return p;
}

// A pool allocation that goes back to the pool when the scope ends, unless keep() hands it on.
// (Frees are stream ordered: every user of these buffers runs on the one setup stream.)
template <typename T>
struct AmgScratch {
    nodal_ctx* ctx;
    T* ptr;
    AmgScratch(nodal_ctx* c, size_t count) : ctx(c), ptr(amg_pool<T>(c, count)) {}
    ~AmgScratch() { ctx_pool_free(ctx, ptr); }
    AmgScratch(const AmgScratch&) = delete;
    AmgScratch& operator=(const AmgScratch&) = delete;
    T* keep() { T* p = ptr; ptr = nullptr; return p; }
    operator T*() const { return ptr; }
};

// ------------------------------------------------------------------ the hierarchy (amg.cu builds it, amg_multi.cu reads it)
struct AmgLevel {
    int32_t n = 0;
    int64_t nnz = 0;
    const int32_t* indptr = nullptr;    // CSR of the level operator (level 0: the caller's arrays)
    const int32_t* indices = nullptr;
    const double* data = nullptr;
    bool owned = false;
    nodal_sell* sell = nullptr;
    int32_t nc = 0;                     // rows of the next level (0 on the coarsest)
    int32_t* agg = nullptr;             // [n]  row -> aggregate
    int32_t* pt_ptr = nullptr;          // [>= nc + 1]  members of every aggregate ...
    int32_t* pt_idx = nullptr;          // [n]          ... in increasing row order
    double *b = nullptr, *x = nullptr, *r = nullptr;   // cycle work vectors (b: levels > 0)
};

struct nodal_amg {
    nodal_ctx* ctx = nullptr;
    int device = 0;
    int passes = 2, coarse = 512, maxlevels = 30, rounds = 8, direct_max = 2048;
    double omega = 0.8, scale = 1.8, max_fill = 1.2, max_complexity = 4.0;
    std::vector<AmgLevel> lv;           // lv.back() is the coarsest level
    double* inv = nullptr;              // [nL x nL] inverse of the coarsest operator (or nullptr)
    double *p = nullptr, *q = nullptr, *r = nullptr, *z = nullptr;   // CG vectors
    double* part = nullptr;             // 3 x nparts partial sums + scalars
    int nparts = 0;
    float setup_ms = 0.f;
};

struct AmgCsr {
    int32_t n = 0;
    int64_t nnz = 0;
    const int32_t* indptr = nullptr;
    const int32_t* indices = nullptr;
    const double* data = nullptr;
    bool owned = false;
};
void amg_free_csr(nodal_ctx* ctx, AmgCsr& a);

// One pairwise pass over the rows of A: *agg_out[n] (pool, owned by the caller) and the number
// of aggregates.  Columns >= nown never qualify and `base` offsets the tie-breaking hash
// (amg_core.cuh); the single-GPU setup passes nown = INT32_MAX, base = 0.
int amg_aggregate(nodal_ctx* ctx, int rounds, const AmgCsr& A, int32_t nown, int32_t base,
                  int32_t** agg_out, int32_t* nc_out, cudaStream_t st);
// Members of the nc aggregates (CSR pattern of P^T), rows in increasing order, by count / scan /
// place / per-aggregate ordering; pool buffers pt_ptr[nc + 1] / pt_idx[n] owned by the caller.
int amg_members(nodal_ctx* ctx, int32_t n, const int32_t* agg, int32_t nc, int32_t** pt_ptr, int32_t** pt_idx,
                cudaStream_t st);
// Rows [0, nc) of P^T A P by merging the member rows of every coarse row (amg_merge_core.cuh):
// A's rows are the fine rows the members refer to, `label[col]` is the coarse column of a fine
// column, columns >= ncol_limit are skipped.  Bit-identical to the sort + in-order sum it replaces.
int amg_galerkin_merge(nodal_ctx* ctx, const AmgCsr& A, const int32_t* pt_ptr, const int32_t* pt_idx, int32_t nc,
                       const int32_t* label, int32_t ncol_limit, AmgCsr* out, cudaStream_t st);

// The merge keeps a coarse row's entries in an insertion-sorted list: linear work per row on
// grid-like operators (10 - 25 entries per coarse row), quadratic on rows that collect hundreds of
// entries (coarse levels of expander-like graphs: 15.8 s instead of 0.13 s of setup on a 4 M-node
// random network).  Those products go through the sort-based builder (same values bit for bit).
static inline bool amg_merge_pays(int64_t fine_nnz, int64_t coarse_rows) {
    return fine_nnz <= 40 * (coarse_rows > 0 ? coarse_rows : 1);
}
