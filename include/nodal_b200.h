/*
 * nodal_b200 -- C ABI of the B200-native MNA hot path (libnodal_b200.so).
 *
 * The reference (EnricoMiccoli/nodal) is pure Python and has no FFI; its de-facto
 * boundary for this path is the Python object surface (Circuit.build_model,
 * nodal/nodal.py:338-398; Circuit.solve, nodal/nodal.py:313-336; the write_*
 * stamp functions, nodal/models.py:13-214).  Each entry point below names the
 * reference code it replaces.  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C symbols, plain pointers and sizes; no torch / C++ types.
 *   - every pointer is a DEVICE pointer supplied (and owned) by the caller unless
 *     its name ends in _h (host).  Nothing passed in is freed by the library.
 *   - `stream` is a cudaStream_t passed as void*; calls that return only a status
 *     are asynchronous on that stream, calls that fill host scalars synchronise it.
 *   - return value: NODAL_OK, or one of the codes below; a message for the last
 *     error of the calling thread is available from nodal_last_error().
 *   - a nodal_ctx owns scratch workspaces for one device; it is not thread safe:
 *     use one ctx per host thread / stream.
 */
#ifndef NODAL_B200_H
#define NODAL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NODAL_ABI_VERSION 1

enum {
    NODAL_OK = 0,
    NODAL_SINGULAR = 1,      /* zero pivot in LU; *info_h = 1-based pivot index            */
    NODAL_NOT_CONVERGED = 2, /* Krylov solver hit maxit; iters / relres are still filled  */
    NODAL_BREAKDOWN = 3,     /* Krylov breakdown (p.Ap <= 0 in CG, zero Arnoldi vector)   */
    NODAL_CUDA_ERROR = 4,    /* CUDA / NCCL failure, see nodal_last_error()               */
    NODAL_BAD_ARG = -1
};

/* component type codes of the struct-of-arrays table (nodal/constants.py:15-18) */
enum { NODAL_T_R = 0, NODAL_T_A = 1, NODAL_T_E = 2, NODAL_T_VCVS = 3, NODAL_T_VCCS = 4,
       NODAL_T_CCVS = 5, NODAL_T_CCCS = 6 };
#define NODAL_GROUND (-1) /* lead / control index of the ground node */
#define NODAL_UNUSED (-2)

typedef struct nodal_ctx nodal_ctx;

int nodal_abi_version(void);
const char* nodal_last_error(void);
/* number of kernels this library has launched so far in this process (graph nodes count
 * once per graph launch) */
uint64_t nodal_launch_count(void);
int nodal_ctx_create(int device, nodal_ctx** out);
int nodal_ctx_destroy(nodal_ctx* ctx);
/* bytes of device scratch currently held by the ctx */
int64_t nodal_ctx_workspace_bytes(nodal_ctx* ctx);

/* ---------------------------------------------------------------- stamping
 * Replaces the loop of Circuit.build_model (nodal/nodal.py:357-390) and the
 * write_R/A/E/VCVS/CCVS/CCCS stamp functions (nodal/models.py:13-214).
 *
 * Reads the component table (one row per component, stamping order) and emits
 * `stride` keyed triples per component into keys/vals (capacity stride*ncomp):
 *   key = (row << colbits) | col, val = contribution.  Right-hand-side
 *   contributions use col == n.  Unused slots get row == n (sorts last).
 * stride must be >= the largest number of entries any present type emits
 * (R 4, A 2, E 5, VCVS/VCCS/CCVS 6, CCCS 5); colbits = bits needed for n.
 * Within-component '=' / '+=' ordering of the reference is resolved here, so
 * the later reduction is a pure in-order sum.
 * c, d, drv and branch may be NULL when the table holds only R and A rows (the columns are
 * then the constants NODAL_UNUSED / -1 and are not read): 17 instead of 33 bytes per component.
 * The same holds for nodal_lu_batched* and nodal_table_select_gather.
 */
int nodal_stamp_coo(nodal_ctx* ctx, int64_t ncomp,
                    const uint8_t* type, const double* value,
                    const int32_t* a, const int32_t* b, const int32_t* c, const int32_t* d,
                    const int32_t* drv, const int32_t* branch,
                    int32_t kcl, int32_t n, int32_t stride, int32_t colbits,
                    uint64_t* keys, double* vals, void* stream);

/* ---------------------------------------------------------------- CSR build
 * Replaces dok_matrix accumulation + G.tocsr() (nodal/nodal.py:349-351,396-397)
 * and the in-place sum_duplicates() spsolve performs (canonical sorted columns).
 *
 * Phase 1: stable LSD radix sort of (keys, vals) [both are clobbered], in-order
 * segmented sum of duplicates (reproduces the reference's summation order bit for
 * bit), removal of exact zeros (DOK semantics), split of the col == n entries
 * into rhs[n] (rhs is fully overwritten).  Returns nnz in *nnz_h (synchronises).
 * Phase 2: copies the result into caller buffers indptr[n+1], indices[nnz],
 * data[nnz].
 */
int nodal_csr_build(nodal_ctx* ctx, int32_t n, int64_t nslots, int32_t colbits,
                    uint64_t* keys, double* vals, double* rhs,
                    int64_t* nnz_h, void* stream);
int nodal_csr_fetch(nodal_ctx* ctx, int32_t n, int64_t nnz,
                    int32_t* indptr, int32_t* indices, double* data, void* stream);
/* nodal_csr_build with the column order chosen: order 0 = sorted (what nodal_csr_build gives and what
 * scipy's spsolve leaves in circuit.G), order 1 = first touch, the order `G.tocsr()` of the reference's DOK
 * matrix has before the solve (nodal/nodal.py:396-397): within a row, columns appear in the order their
 * keys were inserted; a key whose running sum hit exact zero was deleted and counts from its re-insertion.
 * Followed by nodal_csr_fetch as usual.  Values are identical in both orders. */
int nodal_csr_build_ordered(nodal_ctx* ctx, int32_t n, int64_t nslots, int32_t colbits,
                            uint64_t* keys, double* vals, int32_t order, double* rhs, int64_t* nnz_h,
                            void* stream);

/* CSR -> dense row-major n x n (dense mode of build_model, nodal/nodal.py:352-353).
 * G is fully overwritten. */
int nodal_csr_to_dense(nodal_ctx* ctx, int32_t n, const int32_t* indptr, const int32_t* indices,
                       const double* data, double* G, void* stream);
/* Dense scatter-add of the keyed triples with warp-aggregated atomics (fast,
 * summation order not reproducible).  G (n x n) and rhs (n) are overwritten. */
int nodal_coo_to_dense_atomic(nodal_ctx* ctx, int32_t n, int64_t nslots, int32_t colbits,
                              const uint64_t* keys, const double* vals, double* G, double* rhs,
                              void* stream);

/* ---------------------------------------------------------------- sparse kernels */
/* y = A x (CSR, f64 values, i32 indices). */
int nodal_spmv(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
               const int32_t* indices, const double* data, const double* x, double* y,
               void* stream);

/* Solver-private sliced-ELL copy of a CSR matrix (slice height 32).  The handle
 * is owned by the ctx-independent library heap; free with nodal_sell_destroy. */
typedef struct nodal_sell nodal_sell;
int nodal_sell_create(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                      const int32_t* indices, const double* data, nodal_sell** out, void* stream);
int nodal_sell_destroy(nodal_sell* m);
int64_t nodal_sell_padded_nnz(const nodal_sell* m);
int nodal_sell_spmv(nodal_ctx* ctx, const nodal_sell* m, const double* x, double* y, void* stream);

/* Jacobi-preconditioned conjugate gradients, FP64.  Replaces
 * scipy.sparse.linalg.spsolve at nodal/nodal.py:325 for SPD (R / A only) netlists.
 * x holds the initial guess on entry and the solution on exit.  Converged when
 * ||b - A x||_2 <= rtol * ||b||_2 (checked on the true residual at the end).
 * stats_h (optional, 16 doubles): [0] iterations, [1] relres (true), [2] restarts,
 * [3] solve ms (device), [4] setup ms, [5] format (0 csr, 1 sell), [6] stored nnz,
 * [7] SpMV grid size; with NODAL_PCG_PROFILE: [8..10] mean ms of the spmv_dot / update /
 * direction kernels, [11] launches averaged over. */
int nodal_pcg(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
              const int32_t* indices, const double* data, const double* rhs, double* x,
              double rtol, int32_t maxit, int32_t flags,
              int32_t* iters_h, double* relres_h, double* stats_h, void* stream);
#define NODAL_PCG_FORCE_CSR 1   /* do not build the sliced-ELL copy          */
#define NODAL_PCG_NO_GRAPH 2    /* launch kernels directly (debug)           */
#define NODAL_PCG_PROFILE 4     /* direct launches, every kernel bracketed by CUDA events */
#define NODAL_PCG_NO_SCALE 8    /* keep D^-1 as an explicit preconditioner (no S A S pre-scaling) */

/* Restarted GMRES(m) with diagonal (zero-safe) right preconditioning, FP64.
 * Replaces spsolve at nodal/nodal.py:325 when controlled / voltage sources make
 * G non-symmetric. */
int nodal_gmres(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                const int32_t* indices, const double* data, const double* rhs, double* x,
                double rtol, int32_t restart, int32_t maxit,
                int32_t* iters_h, double* relres_h, void* stream);

/* ---------------------------------------------------------------- AMG-preconditioned CG
 * Alternative to nodal_pcg for the same call site (`spsolve(G, A)`, nodal/nodal.py:325) on
 * symmetric positive definite systems: a V(1,1) cycle over pairwise aggregates (csrc/amg.cu)
 * replaces the Jacobi preconditioner, so the iteration count stays nearly flat in n.
 *
 * nodal_amg_create builds the hierarchy for the CSR matrix (device pointers; the arrays must
 * stay alive and unchanged until nodal_amg_destroy).  params is NULL or 8 doubles, 0 = default:
 * [0] pairwise passes per level (2), [1] stop coarsening at this many rows (512), [2] Jacobi
 * damping (0.8), [3] coarse-correction scale (1.8), [4] max levels (30), [5] handshake rounds
 * (8), [6] largest coarsest level that is inverted explicitly (2048), [7] max_fill: coarsening stops
 * when a coarser operator would hold more than this multiple of its parent's entries (1.2) or the
 * operator complexity would pass 4 (graphs that fill in instead of shrinking).
 * nodal_amg_info: level count, rows / nnz per level (up to cap entries), setup time, whether the
 * coarsest level is solved exactly.  nodal_amg_fetch_level copies a level's aggregate map
 * (agg, n entries; not on the coarsest level) and/or CSR arrays to device buffers (NULL = skip).
 * nodal_amg_apply: z = M r, one cycle.  nodal_amg_pcg: solve A x = rhs starting from x;
 * status / iters_h / relres_h as nodal_pcg (relres is the true residual); stats_h (16 doubles or
 * NULL): [0] levels, [1] operator complexity, [2] restarts, [3] solve ms, [4] setup ms,
 * [5] rows of the coarsest level, [6] grid complexity, [7] coarsest level solved exactly. */
typedef struct nodal_amg nodal_amg;
int nodal_amg_create(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                     const int32_t* indices, const double* data, const double* params,
                     nodal_amg** out, void* stream);
int nodal_amg_destroy(nodal_amg* amg);
int nodal_amg_info(const nodal_amg* amg, int32_t cap, int32_t* nlevels, int64_t* rows, int64_t* nnz,
                   double* setup_ms, int32_t* direct);
int nodal_amg_fetch_level(nodal_ctx* ctx, const nodal_amg* amg, int32_t level, int32_t* agg,
                          int32_t* indptr, int32_t* indices, double* data, void* stream);
int nodal_amg_apply(nodal_ctx* ctx, const nodal_amg* amg, const double* r, double* z, void* stream);
int nodal_amg_pcg(nodal_ctx* ctx, nodal_amg* amg, const double* rhs, double* x, double rtol,
                  int32_t maxit, int32_t* iters_h, double* relres_h, double* stats_h, void* stream);

/* ---------------------------------------------------------------- connectivity
 * Connected components of the lead graph (nodes 0..kcl-1 plus ground = node kcl; one edge
 * anode - bnode per component, ground leads are negative indices).  Replaces the breadth-first
 * search is_connected (nodal/nodal.py:88-105) behind the singular-matrix diagnosis
 * (nodal/nodal.py:328-335).  labels (device, kcl + 1 entries, or NULL) receives the smallest
 * node index of every node's component; *ncomponents_h the number of components,
 * *reached_h the number of nodes connected to ground (== kcl + 1 iff the circuit is connected). */
int nodal_connected_components(nodal_ctx* ctx, int64_t ncomp, const int32_t* a, const int32_t* b,
                               int32_t kcl, int32_t* labels, int32_t* ncomponents_h,
                               int32_t* reached_h, void* stream);

/* ---------------------------------------------------------------- voltage-source elimination
 * csrc/sources.cu.  For an R / A / E table whose E rows form a forest (no loop of sources, every
 * branch owned by exactly one E row), the MNA system the reference hands to spsolve
 * (nodal/nodal.py:325) is reduced to an R / A table over one unknown per tree of sources (an SPD
 * weighted Laplacian), solved with the SPD solvers, and expanded back.  Nodes are 0..kcl-1 plus
 * ground = node kcl.
 *
 * nodal_source_forest: erow (be) receives the table rows of the E sources in table order;
 * adj_ptr (kcl + 2) / adj_row (2 be) every node's incident sources ordered by the other node;
 * per node (kcl + 1): rep_row (reduced row of its tree, NODAL_GROUND for ground's tree), offset
 * (potential relative to the tree's root), parent_edge (table row of the source to its parent, -1
 * at a root), depth; roots (kcl) the root node of each reduced row.  info_h (host, 8): [0] E rows,
 * [1] loops of the source graph, [2] branches not owned by exactly one E row, [3] trees, [4] trees
 * without ground, [5] nodes in ground's tree, [6] reduced rows, [7] depth of the forest.  When
 * [1] or [2] is non-zero the per-node outputs are not written. */
int nodal_source_forest(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const double* value,
                        const int32_t* a, const int32_t* b, const int32_t* branch, int32_t kcl, int32_t be,
                        int32_t* erow, int32_t* adj_ptr, int32_t* adj_row, int32_t* rep_row, double* offset,
                        int32_t* parent_edge, int32_t* depth, int32_t* roots, int64_t* info_h, void* stream);
/* The reduced table (kcl = reduced rows, be = 0) in component order: pos (ncomp) receives each
 * component's first output row, *count_h the number of rows; then nodal_source_reduce_table writes
 * them (csrc/sources_core.cuh src_reduce_component gives the rule). */
int nodal_source_reduce_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                             const int32_t* b, int32_t kcl, const int32_t* rep_row, const double* offset,
                             uint32_t* pos, int64_t* count_h, void* stream);
int nodal_source_reduce_table(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const double* value,
                              const int32_t* a, const int32_t* b, int32_t kcl, const int32_t* rep_row,
                              const double* offset, const uint32_t* pos, uint8_t* out_type, double* out_value,
                              int32_t* out_a, int32_t* out_b, void* stream);
/* x (n) = potentials from the reduced solution y, then the source currents from the KCL residual
 * rhs - G [e; 0] of the full MNA system (indptr / indices / data, n rows) summed over the subtree each
 * source cuts off, deepest level first.  *relres_h = ||rhs - G x|| / ||rhs||. */
int nodal_source_expand(nodal_ctx* ctx, int32_t kcl, int32_t n, int32_t nsrc, const int32_t* erow,
                        const int32_t* a, const int32_t* b, const int32_t* branch, const int32_t* adj_ptr,
                        const int32_t* adj_row, const int32_t* rep_row, const double* offset,
                        const int32_t* depth, int32_t max_depth, const double* y, const double* rhs,
                        int64_t nnz, const int32_t* indptr, const int32_t* indices, const double* data,
                        double* x, double* relres_h, void* stream);
/* The stages of nodal_source_expand for the row-partitioned solve, where a rank holds rows [rb, re)
 * of the full MNA matrix (n rows, nnz_full entries in all; indptr rebased to 0, global columns) and
 * the forest of the E-only table (erow / a / b / branch index that table).  They launch the kernels
 * of nodal_source_expand, and the row products take their lanes per row from (n, nnz_full), so the
 * currents are bit-identical to the single-GPU expansion of the same y.
 * nodal_source_potentials: x (n) = potentials from y (all nodes), 0 on the branch rows.
 * nodal_source_tree_rows: for the rank's rows whose node has depth >= 1, in row order: the row, its
 * rhs entry (rhs: the rank's re - rb entries) and (G x)[row]; out_*: re - rb entries capacity,
 * *count_h the number written.
 * nodal_source_currents: the source currents into x[kcl + branch] from the tree rows of all ranks
 * (ntree entries, any order).
 * nodal_source_residual: sums_h[0] = sum (rhs - G x)^2 and sums_h[1] = sum rhs^2 over the rank's
 * rows (block partials added in a fixed order). */
int nodal_source_potentials(nodal_ctx* ctx, int32_t kcl, int32_t n, const int32_t* rep_row, const double* offset,
                            const double* y, double* x, void* stream);
int nodal_source_tree_rows(nodal_ctx* ctx, int32_t kcl, int32_t n, int64_t nnz_full, int32_t rb, int32_t re,
                           const int32_t* depth, const double* rhs, int64_t nnz, const int32_t* indptr,
                           const int32_t* indices, const double* data, const double* x, int32_t* out_row,
                           double* out_rhs, double* out_gx, int64_t* count_h, void* stream);
int nodal_source_currents(nodal_ctx* ctx, int32_t kcl, int32_t nsrc, const int32_t* erow, const int32_t* a,
                          const int32_t* b, const int32_t* branch, const int32_t* adj_ptr, const int32_t* adj_row,
                          const int32_t* depth, int32_t max_depth, int64_t ntree, const int32_t* tree_row,
                          const double* tree_rhs, const double* tree_gx, double* x, void* stream);
int nodal_source_residual(nodal_ctx* ctx, int32_t n, int64_t nnz_full, int32_t rows, const double* rhs, int64_t nnz,
                          const int32_t* indptr, const int32_t* indices, const double* data, const double* x,
                          double* sums_h, void* stream);

/* ---------------------------------------------------------------- dense kernels
 * Blocked FP64 LU with partial pivoting + triangular solves.  Replaces
 * numpy.linalg.solve (LAPACK dgesv) at nodal/nodal.py:327.  G (n x n row-major)
 * is overwritten by its factors; x receives the solution (rhs untouched).
 * NODAL_SINGULAR with *info_h = k (1-based) when the k-th pivot is exactly zero,
 * matching dgesv's info > 0 -> numpy LinAlgError. */
int nodal_lu_solve(nodal_ctx* ctx, int32_t n, double* G, const double* rhs, double* x,
                   int32_t* info_h, void* stream);

/* Measurement aid: the LU's DMMA trailing-update kernel alone, C[M x N] -= A[M x K] B[K x N] (row-major,
 * even leading dimension ld), average ms per launch over `reps` launches (CUDA events on `stream`).
 * Gives the FP64 tensor-pipe figure the dense path's roofline is quoted against. */
int nodal_dgemm_sub_profile(nodal_ctx* ctx, double* C, const double* A, const double* B, int32_t M, int32_t N,
                            int32_t K, int32_t ld, int32_t reps, double* ms_out, void* stream);

/* Batched small systems sharing one topology: for copy s in [0, batch) stamp the
 * table with values[s*ncomp .. +ncomp) and solve the n x n system (n <= 32) with
 * partially pivoted LU in one thread.  x is batch x n row-major; info[s] = 0 or
 * the 1-based index of a zero pivot.  Replaces a loop of Netlist+Circuit+solve
 * over parameter sweeps (config C4). */
int nodal_lu_batched(nodal_ctx* ctx, int64_t batch, int32_t ncomp,
                     const uint8_t* type, const int32_t* a, const int32_t* b,
                     const int32_t* c, const int32_t* d, const int32_t* drv, const int32_t* branch,
                     int32_t kcl, int32_t n, const double* values, double* x, int32_t* info,
                     void* stream);

/* The same with the transposed (structure-of-arrays) layout: values_t is ncomp x batch and x_t is
 * n x batch, system index fastest, so a warp's loads and stores are contiguous.  n <= 8. */
int nodal_lu_batched_soa(nodal_ctx* ctx, int64_t batch, int32_t ncomp,
                         const uint8_t* type, const int32_t* a, const int32_t* b,
                         const int32_t* c, const int32_t* d, const int32_t* drv, const int32_t* branch,
                         int32_t kcl, int32_t n, const double* values_t, double* x_t, int32_t* info,
                         void* stream);

/* ---------------------------------------------------------------- multi-GPU
 * Row-partitioned PCG: rank k owns rows [bounds[k], bounds[k+1]) of the global
 * system as a local CSR whose column indices are GLOBAL.  Halo exchange of the
 * off-rank x entries + scalar all-reduces run over NCCL (dlopen'ed libnccl.so.2).
 * The 128-byte unique id is created on rank 0 and distributed by the caller
 * (torch.distributed broadcast). */
typedef struct nodal_dist nodal_dist;
int nodal_dist_unique_id(uint8_t id_h[128]);
int nodal_dist_create(nodal_ctx* ctx, const uint8_t id_h[128], int32_t rank, int32_t nranks,
                      nodal_dist** out);
/* one rank, no communicator, libnccl not needed: nodal_dist_amg_pcg then is the graph-captured
 * single-GPU AMG-PCG (nodal_dist_pcg needs a communicator) */
int nodal_dist_create_single(nodal_ctx* ctx, nodal_dist** out);
int nodal_dist_destroy(nodal_dist* d);
/* bounds_h[nranks + 1]: row partition, bounds_h[0] = 0, bounds_h[nranks] = n_global (host).
 * indptr is the local row pointer rebased to 0 (length nloc + 1), nnz = indptr[nloc].
 * stats_h as nodal_pcg, plus [12] halo entries received, [13] entries sent per iteration. */
int nodal_dist_pcg(nodal_ctx* ctx, nodal_dist* d, int32_t n_global, const int32_t* bounds_h,
                   int64_t nnz, const int32_t* indptr, const int32_t* indices, const double* data,
                   const double* rhs_local, double* x_local,
                   double rtol, int32_t maxit,
                   int32_t* iters_h, double* relres_h, double* stats_h, void* stream);

/* Several right-hand sides against one hierarchy (many-port equivalent resistance, nodal/equiv.py:31-61
 * generalised): K <= 8 PCG recurrences advanced together, every level operator read once per sweep for all
 * of them.  rhs / x: K vectors of n doubles, one after the other (x: initial guesses in, solutions out);
 * iters_h, relres_h (true residuals), status_h: K entries.  Returns the worst per-system status. */
int nodal_amg_pcg_multi(nodal_ctx* ctx, nodal_amg* amg, int32_t K, const double* rhs, double* x, double rtol,
                        int32_t maxit, int32_t* iters_h, double* relres_h, int32_t* status_h, void* stream);

/* Measurement aid for bench.py's roofline entry: average per-launch time (ms, CUDA events on
 * `stream`, `reps` launches after two warm-up launches) of the level-0 SELL sweeps of the hierarchy:
 * ms_out[0] q = A p with the p.q partial sums, [1] r = b - A x, [2] the damped-Jacobi sweep. */
int nodal_amg_profile_sweeps(nodal_ctx* ctx, nodal_amg* h, int32_t reps, double* ms_out, void* stream);

/* Measurement aid for benchmarks/amg_cycle.py: average per-launch time (ms, as above) of the
 * level-0 kernels of the V-cycle, unfused and fused (needs at least two levels):
 * ms_out[0] jacobi0, [1] residual sweep, [2] prolong, [3] damped-Jacobi sweep,
 * [4] fused residual of the Jacobi start, [5] fused post-smoothing of the prolongated iterate. */
int nodal_amg_profile_cycle(nodal_ctx* ctx, nodal_amg* h, int32_t reps, double* ms_out, void* stream);

/* Row-partitioned assembly: a rank stamps the components that touch one of its rows [rb, re)
 * (the loop of nodal/nodal.py:357-390 restricted to them, order kept, so the rank's rows of G are
 * bit-identical to the single-GPU CSR).  _scan writes the exclusive scan of the selection flags to
 * pos (device, ncomp entries) and the number selected to *count_h; _gather copies the selected rows
 * of the eight columns, in order, into out_* (device, *count_h entries each).  R / A tables only
 * (drv is copied, not renumbered). */
int nodal_table_select_scan(nodal_ctx* ctx, int64_t ncomp, const int32_t* a, const int32_t* b,
                            int32_t rb, int32_t re, uint32_t* pos, int64_t* count_h, void* stream);
int nodal_table_select_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t rb, int32_t re,
                              const uint8_t* type, const double* value, const int32_t* a, const int32_t* b,
                              const int32_t* c, const int32_t* d, const int32_t* drv, const int32_t* branch,
                              uint8_t* out_type, double* out_value, int32_t* out_a, int32_t* out_b,
                              int32_t* out_c, int32_t* out_d, int32_t* out_drv, int32_t* out_branch,
                              void* stream);
/* The same selection for R / A / E tables (_mna_): a component is also selected when it is an E row
 * whose branch row kcl + branch is in [rb, re) -- the rows it writes are its leads' and that one.
 * type and branch must be given.  And by type (_type_): the components whose type is t (the E rows
 * the source forest is built from). */
int nodal_table_select_mna_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                                const int32_t* b, const int32_t* branch, int32_t kcl, int32_t rb, int32_t re,
                                uint32_t* pos, int64_t* count_h, void* stream);
int nodal_table_select_mna_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t kcl, int32_t rb,
                                  int32_t re, const uint8_t* type, const double* value, const int32_t* a,
                                  const int32_t* b, const int32_t* c, const int32_t* d, const int32_t* drv,
                                  const int32_t* branch, uint8_t* out_type, double* out_value, int32_t* out_a,
                                  int32_t* out_b, int32_t* out_c, int32_t* out_d, int32_t* out_drv,
                                  int32_t* out_branch, void* stream);
int nodal_table_select_type_scan(nodal_ctx* ctx, int64_t ncomp, const uint8_t* type, const int32_t* a,
                                 const int32_t* b, int32_t t, uint32_t* pos, int64_t* count_h, void* stream);
int nodal_table_select_type_gather(nodal_ctx* ctx, int64_t ncomp, const uint32_t* pos, int32_t t,
                                   const uint8_t* type, const double* value, const int32_t* a, const int32_t* b,
                                   const int32_t* c, const int32_t* d, const int32_t* drv, const int32_t* branch,
                                   uint8_t* out_type, double* out_value, int32_t* out_a, int32_t* out_b,
                                   int32_t* out_c, int32_t* out_d, int32_t* out_drv, int32_t* out_branch,
                                   void* stream);

/* Row-partitioned aggregation-AMG preconditioned CG (csrc/dist_amg.cu): same partition contract as
 * nodal_dist_pcg, same call it replaces (spsolve, nodal/nodal.py:325, for R / A netlists).  Aggregates
 * never cross the partition; levels with at most params[7] global rows (default 400 000) are gathered
 * and handled by the single-GPU hierarchy replicated on every rank.  params (host, 8 doubles, 0 = default):
 * passes, coarse, omega, scale, maxlevels, rounds, direct_max (as nodal_amg_create), gather_below,
 * max_fill (9 doubles).
 * With one rank it is a graph-captured single-GPU form of nodal_amg_pcg.
 * stats_h (32 doubles): [0] levels, [2] restarts, [3] solve ms, [4] setup ms, [5] coarsest rows,
 * [7] coarsest solved directly, [8] distributed levels, [9] 2 = peer-memory exchanges / 0 = NCCL,
 * [10] kernels per iteration, [11] rows of the first replicated level, [12] halo entries received per
 * cycle, [16 + l] global rows of level l. */
int nodal_dist_amg_pcg(nodal_ctx* ctx, nodal_dist* d, int32_t n_global, const int32_t* bounds_h,
                       int64_t nnz, const int32_t* indptr, const int32_t* indices, const double* data,
                       const double* rhs_local, double* x_local, const double* params,
                       double rtol, int32_t maxit,
                       int32_t* iters_h, double* relres_h, double* stats_h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NODAL_B200_H */
