// Row-partitioned aggregation-AMG preconditioned CG across GPUs (one process per GPU): the
// multi-GPU form of amg.cu, and -- with one rank -- a graph-captured single-GPU form of it.
// Replaces `spsolve(G, A)` (nodal/nodal.py:325) for R / A netlists whose rows are split over ranks.
//
// Rank k owns the contiguous rows [bounds[k], bounds[k+1]) of every level.
//
// Setup, per distributed level (everything on the device; deterministic):
//   * halo plan of the level operator (off-rank columns -> sorted unique list, owners learn what
//     to send: ncclAllGather of counts + grouped ncclSend/ncclRecv of index lists);
//   * two passes of pairwise aggregation over the rank's OWN rows and columns only (amg_core.cuh
//     with nown / base): no aggregate crosses the partition, so coarse rows stay contiguous per
//     owner and need no communication to number (one all-gather of counts);
//   * the aggregate labels of the halo columns come from their owners through the halo plan;
//   * Galerkin product of the rank's rows with GLOBAL coarse column ids through the CSR builder
//     the assembly uses (radix sort + in-order segmented sum): bit-reproducible.
//   Levels with at most `gather_below` global rows are all-gathered once and handled by the
//   single-GPU hierarchy (amg.cu) replicated on every rank: their sweeps cost microseconds, an
//   exchange per sweep would cost more.
// Cycle: V(1,1) damped Jacobi as in amg.cu.  Every sweep of a distributed level is preceded by a
//   halo exchange of the vector it gathers from.  Peer-memory path (default): all such vectors
//   live in one CUDA-IPC-mapped buffer per rank; an exchange is ONE kernel that stores the
//   entries the peers need straight into their halo tails over NVLink, raises a flag in their
//   mailbox and waits for theirs.  The restricted residual of the first replicated level is
//   all-gathered the same way.  NCCL (grouped send/recv, all-gather) is the fallback.
// CG: single-reduction (Chronopoulos-Gear) form, u = M r, w = A u, gamma = r.u, delta = w.u --
//   one all-reduce per iteration through the mailbox (rank-ordered sum: bitwise identical on all
//   ranks, so every rank takes the same stopping decision).  One iteration is one CUDA graph.
// WAR safety of the mailbox / halo tails: every buffer is written at most once between two
// consecutive all-reduces, and a rank passes an all-reduce only after every peer has finished
// the kernels that read the previous contents (stream order on the peer).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <memory>
#include <vector>

#include "amg_host.cuh"
#include "dist_common.cuh"
#include "pcg_kernels.cuh"

namespace {

constexpr int DA = 256;
constexpr size_t AMG_HDR = 8192;
constexpr int AMG_SLOTS = 60;
struct AmgMail {
    double red[2][P2P_MAXR][4];                       // [parity][source rank] = {v0, v1, v2, v3}
    unsigned long long rtag[2][P2P_MAXR];             // tag of red[parity][source]
    unsigned long long flag[AMG_SLOTS][P2P_MAXR];     // exchange `slot` number `tag` from that rank has landed
    unsigned long long cnt[AMG_SLOTS];                // exchanges of `slot` this rank has completed
    unsigned int ticket[AMG_SLOTS];                   // last-CTA election of a multi-CTA exchange
    unsigned long long rseq;                          // all-reduces this rank has completed
    unsigned long long err;
};
static_assert(sizeof(AmgMail) <= AMG_HDR, "mailbox must fit the header");

#define GRID_LOOP(i, n)                                                                \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)(n); \
         i += (int64_t)gridDim.x * blockDim.x)

// ------------------------------------------------------------------ halo discovery kernels
__global__ void __launch_bounds__(DA)
da_flag_external_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re, u32* __restrict__ flag) {
    GRID_LOOP(i, nnz) { const int32_t c = cols[i]; flag[i] = (c < rb || c >= re) ? 1u : 0u; }
}
__global__ void __launch_bounds__(DA)
da_compact_external_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re,
                           const u32* __restrict__ pos, u64* __restrict__ keys) {
    GRID_LOOP(i, nnz) { const int32_t c = cols[i]; if (c < rb || c >= re) keys[pos[i]] = (u64)(u32)c; }
}
__global__ void __launch_bounds__(DA)
da_unique_flag_kernel(int64_t m, const u64* __restrict__ keys, u32* __restrict__ flag) {
    GRID_LOOP(i, m) flag[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}
__global__ void __launch_bounds__(DA)
da_unique_compact_kernel(int64_t m, const u64* __restrict__ keys, const u32* __restrict__ pos, int32_t* __restrict__ halo) {
    GRID_LOOP(i, m) if (i == 0 || keys[i] != keys[i - 1]) halo[pos[i]] = (int32_t)keys[i];
}
// global column -> local layout [owned | halo]
__global__ void __launch_bounds__(DA)
da_remap_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re,
                const int32_t* __restrict__ halo, int32_t nhalo, int32_t* __restrict__ out) {
    const int32_t nloc = re - rb;
    GRID_LOOP(i, nnz) {
        const int32_t c = cols[i];
        if (c >= rb && c < re) { out[i] = c - rb; continue; }
        int lo = 0, hi = nhalo - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (halo[mid] < c) lo = mid + 1; else hi = mid;
        }
        out[i] = nloc + lo;
    }
}
__global__ void __launch_bounds__(DA)
da_rebase_kernel(int64_t m, int32_t* __restrict__ idx, int32_t rb) { GRID_LOOP(i, m) idx[i] -= rb; }
__global__ void __launch_bounds__(DA)
da_gather_kernel(int64_t m, const int32_t* __restrict__ idx, const double* __restrict__ src, double* __restrict__ dst) {
    GRID_LOOP(i, m) dst[i] = src[idx[i]];
}

// ------------------------------------------------------------------ setup kernels
// labels of the rank's own rows as doubles (exact below 2^53) so they travel through the halo plan
__global__ void __launch_bounds__(DA)
da_labels_kernel(int32_t n, const int32_t* __restrict__ comp, int32_t first, double* __restrict__ lab) {
    GRID_LOOP(i, n) lab[i] = (double)(first + comp[i]);
}
// keys of the local-local block only (pass 2 aggregates inside the rank): entries with a halo
// column become padding (row == nc)
__global__ void __launch_bounds__(DA)
da_relabel_local_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ lcols,
                        const double* __restrict__ data, const int32_t* __restrict__ agg, int32_t nown,
                        int32_t nc, int cb, u64* __restrict__ keys, double* __restrict__ vals) {
    GRID_LOOP(i, n) {
        const u64 hi = (u64)agg[i] << cb;
        const int32_t e = indptr[i + 1];
        for (int32_t p = indptr[i]; p < e; ++p) {
            const int32_t c = lcols[p];
            keys[p] = c < nown ? (hi | (u64)agg[c]) : ((u64)nc << cb);
            vals[p] = data[p];
        }
    }
}
// keys of the rank's rows of P^T A P with global coarse ids (lab covers [owned | halo])
__global__ void __launch_bounds__(DA)
da_relabel_global_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ lcols,
                         const double* __restrict__ data, const double* __restrict__ lab, int cb,
                         u64* __restrict__ keys, double* __restrict__ vals) {
    GRID_LOOP(i, n) {
        const u64 hi = (u64)(int64_t)lab[i] << cb;
        const int32_t e = indptr[i + 1];
        for (int32_t p = indptr[i]; p < e; ++p) {
            keys[p] = hi | (u64)(int64_t)lab[lcols[p]];
            vals[p] = data[p];
        }
    }
}
__global__ void __launch_bounds__(DA)
da_labels_to_i32_kernel(int32_t n, const double* __restrict__ lab, int32_t* __restrict__ out) {
    GRID_LOOP(i, n) out[i] = (int32_t)lab[i];
}
__global__ void __launch_bounds__(DA)
da_slice_indptr_kernel(int32_t nloc, const int32_t* __restrict__ src, int32_t* __restrict__ dst) {
    const int32_t first = src[0];
    GRID_LOOP(i, (int64_t)nloc + 1) dst[i] = src[i] - first;
}
// global indptr of the gathered operator: piece of rank o starts at row bounds[o], entry offset[o]
__global__ void __launch_bounds__(DA)
da_offset_indptr_kernel(int32_t count, int32_t* __restrict__ indptr, int32_t add) {
    GRID_LOOP(i, count) indptr[i] += add;
}
__global__ void da_set_i32_kernel(int32_t* p, int32_t v) { if (threadIdx.x == 0 && blockIdx.x == 0) *p = v; }

// ------------------------------------------------------------------ peer-memory kernels
// Halo exchange of one [owned | halo] vector: every CTA stores its share of the entries the
// peers need into their halo tails; the CTA that finishes last raises this rank's flag in the
// peers' mailboxes and waits for theirs.  mode 1 = all-gather: this rank's `nown` owned entries
// of `src` go to offset dest_off[o] of every rank's copy of the vector (its own included).
__global__ void __launch_bounds__(1024)
da_exchange_kernel(const PcgDev* __restrict__ dev, int slot, int R, int me, long long voff,
                   const double* __restrict__ src, const int32_t* __restrict__ send_idx,
                   const int32_t* __restrict__ send_off, const long long* __restrict__ dest_off,
                   const int32_t* __restrict__ need_cnt, char* const* __restrict__ peer, int mode, int32_t nown) {
    __shared__ int s_last;
    __shared__ unsigned long long s_tag;
    if (dev && block_done(&dev->done)) return;
    AmgMail* mine = reinterpret_cast<AmgMail*>(peer[me]);
    if (threadIdx.x == 0) s_tag = *reinterpret_cast<volatile unsigned long long*>(&mine->cnt[slot]) + 1;
    __syncthreads();
    const unsigned long long tag = s_tag;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gstride = (int64_t)gridDim.x * blockDim.x;
    if (mode == 0) {
        for (int o = 0; o < R; ++o) {
            if (o == me) continue;
            const int b = send_off[o], e = send_off[o + 1];
            double* dst = reinterpret_cast<double*>(peer[o] + voff) + dest_off[o];
            for (int64_t j = b + gtid; j < e; j += gstride) dst[j - b] = src[send_idx[j]];
        }
    } else {
        for (int o = 0; o < R; ++o) {
            double* dst = reinterpret_cast<double*>(peer[o] + voff) + dest_off[o];
            for (int64_t j = gtid; j < nown; j += gstride) dst[j] = src[j];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();   // cumulative: covers the whole CTA's local and remote stores
        const unsigned int t = atomicAdd(&mine->ticket[slot], 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) mine->ticket[slot] = 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence_system();
    if (threadIdx.x < R && threadIdx.x != me) {
        const bool sends = mode == 1 ? nown > 0 : send_off[threadIdx.x + 1] > send_off[threadIdx.x];
        if (sends) st_sys_u64(&reinterpret_cast<AmgMail*>(peer[threadIdx.x])->flag[slot][me], tag);
        if (need_cnt[threadIdx.x] > 0) {
            const long long t0 = clock64();
            while (ld_sys_u64(&mine->flag[slot][threadIdx.x]) < tag) {
                if (clock64() - t0 > P2P_SPIN_LIMIT) { mine->err = 1; break; }
            }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) mine->cnt[slot] = tag;
}

// ------------------------------------------------------------------ CG kernels (single-reduction form)
// SC holds two parity slots {gamma, delta, rr, alpha}; alpha == 0 in the previous slot marks the
// first iteration after a (re)start.
__global__ void __launch_bounds__(DA)
acg_vector_kernel(PcgDev* __restrict__ dev, int32_t n, double* __restrict__ cur, const double* __restrict__ prev,
                  double* __restrict__ x, double* __restrict__ r, double* __restrict__ p, double* __restrict__ s,
                  const double* __restrict__ u, const double* __restrict__ w, double* __restrict__ part_rr) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    const double g = cur[0], dl = cur[1], rr = cur[2];
    const double gp = prev[0], ap = prev[3];
    const bool conv = rr <= dev->tol2;
    double beta = 0.0, den = dl;
    if (ap != 0.0) { beta = g / gp; den = dl - beta * g / ap; }
    const double alpha = g / den;
    const bool bad = !(den > 0.0) || !(rr == rr) || !(g == g);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        dev->rr = rr;
        if (conv) { dev->done = 1; dev->status = NODAL_OK; }
        else if (bad) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
        else { dev->iters = dev->iters + 1; cur[3] = alpha; }
    }
    if (conv || bad) return;
    double lrr = 0.0;
    // ten streams (p, s, r, x read + written, u, w read): 16-byte accesses
    const int64_t n2 = n >> 1;
    double2* x2 = reinterpret_cast<double2*>(x);
    double2* r2 = reinterpret_cast<double2*>(r);
    double2* p2 = reinterpret_cast<double2*>(p);
    double2* s2 = reinterpret_cast<double2*>(s);
    const double2* u2 = reinterpret_cast<const double2*>(u);
    const double2* w2 = reinterpret_cast<const double2*>(w);
    GRID_LOOP(i, n2) {
        double2 pv = p2[i], sv = s2[i], rv = r2[i], xv = x2[i];
        const double2 uv = u2[i], wv = w2[i];
        pv.x = fma(beta, pv.x, uv.x);   pv.y = fma(beta, pv.y, uv.y);
        sv.x = fma(beta, sv.x, wv.x);   sv.y = fma(beta, sv.y, wv.y);
        rv.x = fma(-alpha, sv.x, rv.x); rv.y = fma(-alpha, sv.y, rv.y);
        xv.x = fma(alpha, pv.x, xv.x);  xv.y = fma(alpha, pv.y, xv.y);
        p2[i] = pv; s2[i] = sv; r2[i] = rv; x2[i] = xv;
        lrr = fma(rv.x, rv.x, lrr);
        lrr = fma(rv.y, rv.y, lrr);
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t i = n - 1;
        const double pv = fma(beta, p[i], u[i]);
        const double sv = fma(beta, s[i], w[i]);
        const double rv = fma(-alpha, sv, r[i]);
        p[i] = pv; s[i] = sv; r[i] = rv;
        x[i] = fma(alpha, pv, x[i]);
        lrr = fma(rv, rv, lrr);
    }
    lrr = block_sum(lrr, sm);
    if (threadIdx.x == 0) part_rr[blockIdx.x] = lrr;
}

// w = A u (SELL-32, one warp per slice) + partial sums of r.u and w.u
template <class A>
__global__ void __launch_bounds__(DA, 5)
acg_spmv_dots_kernel(int32_t n, int32_t nslices, const u32* __restrict__ slice_w, A a0, const double* __restrict__ u, const double* __restrict__ r,
                     double* __restrict__ w, double* __restrict__ part_g, double* __restrict__ part_d) {
    __shared__ double sm[40];
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double lg = 0.0, ld = 0.0;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int wd = (int)(slice_w[s + 1] - w0);
        const int64_t row = s * 32 + lane;
        const double acc = sell_row_dot(a, (int64_t)w0 * 32 + lane, row, wd, u);
        if (row < n) {
            const double uv = __ldg(&u[row]);
            w[row] = acc;
            lg = fma(r[row], uv, lg);
            ld = fma(acc, uv, ld);
        }
    }
    lg = block_sum(lg, sm);
    ld = block_sum(ld, sm);
    if (threadIdx.x == 0) { part_g[blockIdx.x] = lg; part_d[blockIdx.x] = ld; }
}

// p = s = 0 ; partial sums of r.r and b.b (r = b - A x was written by the residual sweep)
__global__ void __launch_bounds__(DA)
acg_start_kernel(int32_t n, const double* __restrict__ b, const double* __restrict__ r,
                 double* __restrict__ p, double* __restrict__ s, double* __restrict__ part_rr, double* __restrict__ part_bb) {
    __shared__ double sm[40];
    double lrr = 0.0, lbb = 0.0;
    GRID_LOOP(i, n) {
        const double bv = b[i], rv = r[i];
        p[i] = 0.0; s[i] = 0.0;
        lrr = fma(rv, rv, lrr);
        lbb = fma(bv, bv, lbb);
    }
    lrr = block_sum(lrr, sm);
    lbb = block_sum(lbb, sm);
    if (threadIdx.x == 0) { part_rr[blockIdx.x] = lrr; part_bb[blockIdx.x] = lbb; }
}

// One CTA: out[0..3] = {sum a, sum b, sum c, sum d} over this rank's partials, then summed over
// the ranks through the mailboxes (rank order -> bitwise identical everywhere).  mail == nullptr:
// local sums only (one rank, or the NCCL path which all-reduces `out` afterwards).
__global__ void __launch_bounds__(DA)
acg_allreduce_kernel(PcgDev* __restrict__ dev, int check_done, const double* __restrict__ a, int na,
                     const double* __restrict__ b, int nb, const double* __restrict__ c, int nc,
                     const double* __restrict__ d4, int nd, int R, int me, char* const* __restrict__ peer,
                     int use_mail, double* __restrict__ out, int enforce_maxit) {
    __shared__ double sm[40];
    __shared__ int s_timeout;
    if (check_done && block_done(&dev->done)) return;
    const double va = a ? reduce_partials(a, na, sm) : 0.0;
    const double vb = b ? reduce_partials(b, nb, sm) : 0.0;
    const double vc = c ? reduce_partials(c, nc, sm) : 0.0;
    const double vd = d4 ? reduce_partials(d4, nd, sm) : 0.0;
    if (!use_mail) {
        if (threadIdx.x == 0) {
            out[0] = va; out[1] = vb; out[2] = vc; out[3] = vd;
            if (enforce_maxit && dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        }
        return;
    }
    AmgMail* mine = reinterpret_cast<AmgMail*>(peer[me]);
    const unsigned long long s0 = *reinterpret_cast<volatile unsigned long long*>(&mine->rseq);
    const unsigned long long tag = s0 + 1;
    const int par = (int)(s0 & 1ull);
    if (threadIdx.x == 0) s_timeout = 0;
    __syncthreads();
    if (threadIdx.x < R) {
        AmgMail* m = reinterpret_cast<AmgMail*>(peer[threadIdx.x]);
        volatile double* slot = m->red[par][me];
        slot[0] = va; slot[1] = vb; slot[2] = vc; slot[3] = vd;
        __threadfence_system();
        st_sys_u64(&m->rtag[par][me], tag);
        const long long t0 = clock64();
        while (ld_sys_u64(&mine->rtag[par][threadIdx.x]) != tag) {
            if (clock64() - t0 > P2P_SPIN_LIMIT) { s_timeout = 1; break; }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_timeout) {
            dev->done = 1; dev->status = NODAL_CUDA_ERROR; mine->err = 1;
        } else {
            double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
            for (int t = 0; t < R; ++t) {
                const volatile double* slot = mine->red[par][t];
                t0 += slot[0]; t1 += slot[1]; t2 += slot[2]; t3 += slot[3];
            }
            out[0] = t0; out[1] = t1; out[2] = t2; out[3] = t3;
            mine->rseq = tag;
            if (enforce_maxit && dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        }
    }
}

// after the start all-reduce: SC[0..3] = {gamma, delta, rr, bb}
__global__ void acg_scalars_kernel(PcgDev* dev, double* SC, double rtol, int maxit, int first) {
    if (threadIdx.x != 0) return;
    const double rr = SC[2], bb = SC[3];
    if (first) {
        dev->bb = bb;
        dev->tol2 = rtol * rtol * bb;
        dev->iters = 0;
        dev->maxit = maxit;
    }
    SC[3] = 0.0;       // alpha of parity 0 (written by the first vector pass)
    SC[4] = 1.0;       // gamma_{-1}
    SC[7] = 0.0;       // alpha_{-1} == 0 marks "first iteration"
    dev->rr = rr;
    dev->status = NODAL_OK;
    dev->done = 0;
    if (rr <= dev->tol2) dev->done = 1;
    else if (dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
    else if (!(rr == rr)) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
}

// ------------------------------------------------------------------ host side
struct Halo {
    int32_t nloc = 0, nhalo = 0;
    int64_t send_total = 0;
    int32_t* halo = nullptr;              // dev [nhalo] sorted global column ids
    int32_t* send_idx = nullptr;          // dev [send_total] local rows, grouped by destination
    double* send_buf = nullptr;           // dev [send_total] (NCCL path staging)
    std::vector<int32_t> need_from, need_off, send_cnt, send_off, cnt;   // host; cnt[s * R + o]: s needs from o
    int32_t* send_off_dev = nullptr;      // [R + 1]
    int32_t* need_cnt_dev = nullptr;      // [R]
    long long* dest_off_dev = nullptr;    // [R] where my block starts inside rank o's vector
    int32_t ext_len = 0;                  // nloc + nhalo
};

struct DLevel {
    std::vector<int32_t> bounds;          // [R + 1] row partition of this level
    int32_t nloc = 0, row0 = 0, nglob = 0;
    AmgCsr A;                             // local rows, GLOBAL columns
    int32_t* lcols = nullptr;             // [nnz] columns in the local layout [owned | halo]
    Halo halo;
    nodal_sell* sell = nullptr;
    int32_t* agg = nullptr;               // [nloc] row -> local coarse row
    int32_t nc = 0;                       // local coarse rows
    int32_t* pt_ptr = nullptr;
    int32_t* pt_idx = nullptr;
    double* b = nullptr;                  // [nloc] right-hand side of the level (levels > 0)
    double* x = nullptr;                  // [ext]  in the exchange buffer
    double* r = nullptr;                  // [ext]  residual, then the corrected iterate
    long long x_off = 0, r_off = 0;       // byte offsets of x / r inside the exchange buffer
    int64_t slot_len = 0;                 // doubles reserved per vector (max over ranks)
};

struct Solver {
    nodal_ctx* ctx = nullptr;
    nodal_dist* d = nullptr;
    int R = 1, me = 0;
    cudaStream_t st = nullptr;
    bool p2p = false;
    char* base = nullptr;                 // exchange buffer of this rank (peer-mapped on the p2p path)
    char** peer_dev = nullptr;
    std::vector<void*> owned;             // pool buffers released at the end
    std::vector<DLevel> lv;               // distributed levels (lv[0]: the finest)
    nodal_amg* rep = nullptr;             // replicated hierarchy below the last distributed level
    AmgCsr repA;                          // its finest operator (gathered)
    std::vector<int32_t> rep_bounds;      // row partition of the first replicated level
    int32_t rep_n = 0;
    double *bfull = nullptr, *xfull = nullptr;   // replicated rhs / solution of that level
    long long bfull_off = 0;
    long long* gather_dest_dev = nullptr; // [R] all equal: rep_bounds[me]
    int32_t* gather_need_dev = nullptr;   // [R] rows of every rank at the gathered level
    double* gather_stage = nullptr;       // NCCL path: R * gmax staging
    int32_t gmax = 0;
    double omega = 0.8, scale = 1.8, max_fill = 1.2, max_complexity = 4.0;
    double nnz_k_fine = 0.0, nnz_k_total = 0.0;      // entries (in units of 1024) of level 0 / of all levels so far
    bool sorted_galerkin = getenv("NODAL_AMG_SORT_GALERKIN") != nullptr;   // round-2 first version: sort-based products
    int passes = 2, rounds = 8, maxlevels = 30;
    int64_t gather_below = 400000;
    double params_rep[8] = {0};
    unsigned long long launches_exchange = 0;
    int64_t halo_total = 0;

    template <typename T>
    T* alloc(size_t count) {
        T* p = amg_pool<T>(ctx, count);
        if (p) owned.push_back(p);
        return p;
    }
};

int exchange_nccl(Solver& S, const Halo& H, double* v, cudaStream_t sx) {
    const int R = S.R, me = S.me;
    if (R == 1) return NODAL_OK;
    if (H.send_total) {
        da_gather_kernel<<<amg_rows_grid(S.ctx, H.send_total), DA, 0, sx>>>(H.send_total, H.send_idx, v, H.send_buf);
        KERNEL_CHECK();
    }
    NCCL_TRY(g_nccl.GroupStart());
    for (int o = 0; o < R; ++o) {
        if (o == me) continue;
        if (H.send_cnt[o]) NCCL_TRY(g_nccl.Send(H.send_buf + H.send_off[o], H.send_cnt[o], ncclFloat64, o, S.d->comm, sx));
        if (H.need_from[o]) NCCL_TRY(g_nccl.Recv(v + H.nloc + H.need_off[o], H.need_from[o], ncclFloat64, o, S.d->comm, sx));
    }
    NCCL_TRY(g_nccl.GroupEnd());
    return NODAL_OK;
}

// Halo exchange of the [owned | halo] vector at byte offset `voff` of the exchange buffer.
int exchange(Solver& S, const PcgDev* dev, int slot, const Halo& H, long long voff, cudaStream_t sx) {
    if (S.R == 1) return NODAL_OK;
    double* v = reinterpret_cast<double*>(S.base + voff);
    if (!S.p2p) return exchange_nccl(S, H, v, sx);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(16, (H.send_total + 4095) / 4096));
    da_exchange_kernel<<<grid, 1024, 0, sx>>>(dev, slot, S.R, S.me, voff, v, H.send_idx, H.send_off_dev, H.dest_off_dev,
                                              H.need_cnt_dev, S.peer_dev, 0, 0);
    KERNEL_CHECK();
    return NODAL_OK;
}

// Halo plan of a local operator with global columns; also the columns in the local layout.
int build_halo(Solver& S, DLevel& L) {
    nodal_ctx* ctx = S.ctx;
    cudaStream_t st = S.st;
    const int R = S.R, me = S.me;
    const int32_t rb = L.bounds[me], re = L.bounds[me + 1];
    const int64_t nnz = L.A.nnz;
    Halo& H = L.halo;
    H.nloc = L.nloc;
    const size_t need = align_up((size_t)std::max<int64_t>(nnz, 1) * 4, 256) * 2 +
                        align_up((size_t)std::max<int64_t>(nnz, 1) * 8, 256) * 4 +
                        radix_sort_scratch_bytes(std::max<int64_t>(nnz, 1)) +
                        2 * scan_scratch_bytes(std::max<int64_t>(nnz, 1)) + (1 << 16);
    NODAL_TRY(ctx_reserve(ctx, need));
    u32* flag = carve<u32>(ctx, (size_t)std::max<int64_t>(nnz, 1));
    u32* tot = carve<u32>(ctx, 16);
    if (!flag || !tot) return NODAL_CUDA_ERROR;
    u32* host_tot = reinterpret_cast<u32*>(ctx->pinned);
    const int gnz = amg_rows_grid(ctx, nnz);
    int64_t next = 0, nhalo = 0;
    if (nnz > 0 && R > 1) {
        da_flag_external_kernel<<<gnz, DA, 0, st>>>(nnz, L.A.indices, rb, re, flag);
        KERNEL_CHECK();
        const size_t mark = ctx->arena_used;
        NODAL_TRY(scan_exclusive_u32(ctx, flag, flag, nnz, tot, st));
        ctx->arena_used = mark;
        CUDA_TRY(cudaMemcpyAsync(host_tot, tot, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        next = host_tot[0];
    }
    if (next > 0) {
        u64* keys = carve<u64>(ctx, (size_t)next);
        u64* vals = carve<u64>(ctx, (size_t)next);
        u64* keys_alt = carve<u64>(ctx, (size_t)next);
        u64* vals_alt = carve<u64>(ctx, (size_t)next);
        u32* uflag = carve<u32>(ctx, (size_t)next);
        if (!keys || !vals || !keys_alt || !vals_alt || !uflag) return NODAL_CUDA_ERROR;
        da_compact_external_kernel<<<gnz, DA, 0, st>>>(nnz, L.A.indices, rb, re, flag, keys);
        KERNEL_CHECK();
        const int bits = amg_bit_length(L.nglob);
        bool in_alt = false;
        const size_t mark = ctx->arena_used;
        NODAL_TRY(radix_sort_pairs(ctx, keys, vals, keys_alt, vals_alt, next, bits, &in_alt, st));
        ctx->arena_used = mark;
        const u64* sk = in_alt ? keys_alt : keys;
        da_unique_flag_kernel<<<amg_rows_grid(ctx, next), DA, 0, st>>>(next, sk, uflag);
        KERNEL_CHECK();
        NODAL_TRY(scan_exclusive_u32(ctx, uflag, uflag, next, tot, st));
        ctx->arena_used = mark;
        CUDA_TRY(cudaMemcpyAsync(host_tot, tot, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        nhalo = host_tot[0];
        H.halo = S.alloc<int32_t>((size_t)nhalo);
        if (!H.halo) return NODAL_CUDA_ERROR;
        da_unique_compact_kernel<<<amg_rows_grid(ctx, next), DA, 0, st>>>(next, sk, uflag, H.halo);
        KERNEL_CHECK();
    }
    H.nhalo = (int32_t)nhalo;
    H.ext_len = L.nloc + H.nhalo;
    S.halo_total += nhalo;
    L.lcols = S.alloc<int32_t>((size_t)std::max<int64_t>(nnz, 1));
    if (!L.lcols) return NODAL_CUDA_ERROR;
    if (nnz > 0) {
        da_remap_kernel<<<gnz, DA, 0, st>>>(nnz, L.A.indices, rb, re, H.halo, H.nhalo, L.lcols);
        KERNEL_CHECK();
    }
    H.need_from.assign(R, 0); H.need_off.assign(R + 1, 0);
    H.send_cnt.assign(R, 0); H.send_off.assign(R + 1, 0);
    H.cnt.assign((size_t)R * R, 0);
    L.slot_len = (int64_t)align_up((size_t)H.ext_len + 2, 32);
    if (R == 1) return NODAL_OK;
    // ---- who needs what (host bookkeeping of <= R counts)
    std::vector<int32_t> halo_h((size_t)nhalo);
    if (nhalo) CUDA_TRY(cudaMemcpyAsync(halo_h.data(), H.halo, sizeof(int32_t) * (size_t)nhalo, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    {
        int o = 0;
        for (int64_t i = 0; i < nhalo; ++i) {
            while (halo_h[i] >= L.bounds[o + 1]) ++o;
            H.need_from[o]++;
        }
        for (int o2 = 0; o2 < R; ++o2) H.need_off[o2 + 1] = H.need_off[o2] + H.need_from[o2];
    }
    const int W = R + 1;       // per rank: R counts + its vector length
    int32_t* cnt_dev = S.alloc<int32_t>((size_t)W * (R + 1));
    if (!cnt_dev) return NODAL_CUDA_ERROR;
    std::vector<int32_t> mine_row(W, 0);
    for (int o = 0; o < R; ++o) mine_row[o] = H.need_from[o];
    mine_row[R] = (int32_t)(L.slot_len / 32);
    CUDA_TRY(cudaMemcpyAsync(cnt_dev + (size_t)W * R, mine_row.data(), sizeof(int32_t) * W, cudaMemcpyHostToDevice, st));
    NCCL_TRY(g_nccl.AllGather(cnt_dev + (size_t)W * R, cnt_dev, W, ncclInt32, S.d->comm, st));
    std::vector<int32_t> gathered((size_t)W * R);
    CUDA_TRY(cudaMemcpyAsync(gathered.data(), cnt_dev, sizeof(int32_t) * (size_t)W * R, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    int64_t max_units = 0;
    for (int s2 = 0; s2 < R; ++s2) {
        for (int o = 0; o < R; ++o) H.cnt[(size_t)s2 * R + o] = gathered[(size_t)s2 * W + o];
        max_units = std::max<int64_t>(max_units, gathered[(size_t)s2 * W + R]);
    }
    L.slot_len = max_units * 32;
    for (int s = 0; s < R; ++s) H.send_cnt[s] = H.cnt[(size_t)s * R + me];
    for (int s = 0; s < R; ++s) H.send_off[s + 1] = H.send_off[s] + H.send_cnt[s];
    H.send_total = H.send_off[R];
    H.send_idx = S.alloc<int32_t>((size_t)std::max<int64_t>(H.send_total, 1));
    H.send_buf = S.alloc<double>((size_t)std::max<int64_t>(H.send_total, 1));
    if (!H.send_idx || !H.send_buf) return NODAL_CUDA_ERROR;
    NCCL_TRY(g_nccl.GroupStart());
    for (int o = 0; o < R; ++o) {
        if (o == me) continue;
        if (H.need_from[o]) NCCL_TRY(g_nccl.Send(H.halo + H.need_off[o], H.need_from[o], ncclInt32, o, S.d->comm, st));
        if (H.send_cnt[o]) NCCL_TRY(g_nccl.Recv(H.send_idx + H.send_off[o], H.send_cnt[o], ncclInt32, o, S.d->comm, st));
    }
    NCCL_TRY(g_nccl.GroupEnd());
    if (H.send_total) {
        da_rebase_kernel<<<amg_rows_grid(ctx, H.send_total), DA, 0, st>>>(H.send_total, H.send_idx, rb);
        KERNEL_CHECK();
    }
    // device tables of the push kernel
    std::vector<long long> dest_off(R, 0);
    for (int o = 0; o < R; ++o) {
        long long off = L.bounds[o + 1] - L.bounds[o];                       // peer's owned part
        for (int o2 = 0; o2 < me; ++o2) off += H.cnt[(size_t)o * R + o2];    // blocks of lower-ranked owners
        dest_off[o] = off;
    }
    H.send_off_dev = S.alloc<int32_t>((size_t)R + 1);
    H.need_cnt_dev = S.alloc<int32_t>((size_t)R);
    H.dest_off_dev = S.alloc<long long>((size_t)R);
    if (!H.send_off_dev || !H.need_cnt_dev || !H.dest_off_dev) return NODAL_CUDA_ERROR;
    CUDA_TRY(cudaMemcpyAsync(H.send_off_dev, H.send_off.data(), sizeof(int32_t) * (size_t)(R + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(H.need_cnt_dev, H.need_from.data(), sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(H.dest_off_dev, dest_off.data(), sizeof(long long) * (size_t)R, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return NODAL_OK;
}

// counts of every rank -> bounds (host); one tiny all-gather
int gather_counts(Solver& S, int32_t mine, std::vector<int32_t>& bounds) {
    const int R = S.R;
    bounds.assign(R + 1, 0);
    if (R == 1) { bounds[1] = mine; return NODAL_OK; }
    int32_t* dev = S.alloc<int32_t>((size_t)R + 1);
    if (!dev) return NODAL_CUDA_ERROR;
    CUDA_TRY(cudaMemcpyAsync(dev + R, &mine, sizeof(int32_t), cudaMemcpyHostToDevice, S.st));
    NCCL_TRY(g_nccl.AllGather(dev + R, dev, 1, ncclInt32, S.d->comm, S.st));
    std::vector<int32_t> h(R);
    CUDA_TRY(cudaMemcpyAsync(h.data(), dev, sizeof(int32_t) * (size_t)R, cudaMemcpyDeviceToHost, S.st));
    CUDA_TRY(cudaStreamSynchronize(S.st));
    for (int o = 0; o < R; ++o) bounds[o + 1] = bounds[o] + h[o];
    return NODAL_OK;
}

// CSR of sorted keyed triples through the assembly's builder; rows [row_first, row_first + nrows)
// of the n_shape-row result are returned with a rebased row pointer (pool buffers).
int build_rows(Solver& S, int32_t n_shape, int64_t nslots, int cb, u64* keys, double* vals, int32_t row_first,
               int32_t nrows, AmgCsr* out) {
    nodal_ctx* ctx = S.ctx;
    cudaStream_t st = S.st;
    AmgScratch<double> rhs(ctx, (size_t)n_shape + 1);
    if (!rhs.ptr) return NODAL_CUDA_ERROR;
    int64_t nnz = 0;
    NODAL_TRY(nodal_csr_build(ctx, n_shape, nslots, cb, reinterpret_cast<uint64_t*>(keys), vals, rhs, &nnz, st));
    AmgScratch<int32_t> ip_full(ctx, (size_t)n_shape + 1), ix(ctx, (size_t)std::max<int64_t>(nnz, 1));
    AmgScratch<double> dv(ctx, (size_t)std::max<int64_t>(nnz, 1));
    if (!ip_full.ptr || !ix.ptr || !dv.ptr) return NODAL_CUDA_ERROR;
    NODAL_TRY(nodal_csr_fetch(ctx, n_shape, nnz, ip_full, ix, dv, st));
    out->n = nrows;
    out->nnz = nnz;          // every entry belongs to a row of the slice
    out->owned = true;
    if (row_first == 0 && nrows == n_shape) {
        out->indptr = ip_full.keep();
    } else {
        AmgScratch<int32_t> ip(ctx, (size_t)nrows + 1);
        if (!ip.ptr) return NODAL_CUDA_ERROR;
        da_slice_indptr_kernel<<<amg_rows_grid(ctx, nrows + 1), DA, 0, st>>>(nrows, ip_full.ptr + row_first, ip);
        KERNEL_CHECK();
        out->indptr = ip.keep();
    }
    out->indices = ix.keep();
    out->data = dv.keep();
    return NODAL_OK;
}

// One distributed coarsening step: fills L.agg / L.nc / L.pt_* and returns the next operator.
int coarsen(Solver& S, DLevel& L, AmgCsr* next, std::vector<int32_t>* next_bounds, bool* stalled) {
    nodal_ctx* ctx = S.ctx;
    cudaStream_t st = S.st;
    const int32_t nloc = L.nloc;
    const int64_t nnz = L.A.nnz;
    *stalled = false;
    AmgCsr loc;              // the rank's rows with columns in the local layout
    loc.n = nloc; loc.nnz = nnz; loc.indptr = L.A.indptr; loc.indices = L.lcols; loc.data = L.A.data;
    int32_t* comp = nullptr;
    int32_t ncur = nloc;
    AmgCsr cur = loc;
    int32_t cur_own = nloc, cur_base = L.row0;
    for (int pass = 0; pass < S.passes; ++pass) {
        int32_t* agg = nullptr;
        int32_t nc = 0;
        NODAL_TRY(amg_aggregate(ctx, S.rounds, cur, cur_own, cur_base, &agg, &nc, st));
        if (comp) {
            amg_compose_kernel<<<amg_rows_grid(ctx, nloc), AT, 0, st>>>(nloc, comp, agg);
            KERNEL_CHECK();
        }
        if (pass + 1 < S.passes && !S.sorted_galerkin && amg_merge_pays(cur.nnz, nc)) {
            // operator the next pass aggregates: the local-local block of P^T A P (couplings to
            // other ranks are invisible to the matching, see amg_core.cuh), merged per coarse row
            int32_t *pp = nullptr, *pi = nullptr;
            NODAL_TRY(amg_members(ctx, cur.n, agg, nc, &pp, &pi, st));
            AmgCsr nxt;
            const int rc = amg_galerkin_merge(ctx, cur, pp, pi, nc, agg, cur_own, &nxt, st);
            ctx_pool_free(ctx, pp);
            ctx_pool_free(ctx, pi);
            NODAL_TRY(rc);
            if (cur.owned) amg_free_csr(ctx, cur);
            cur = nxt;
            std::vector<int32_t> ib;
            NODAL_TRY(gather_counts(S, nc, ib));
            cur_own = nc;
            cur_base = ib[S.me];
        } else if (pass + 1 < S.passes) {
            AmgScratch<u64> keys(ctx, (size_t)std::max<int64_t>(cur.nnz, 1));
            AmgScratch<double> vals(ctx, (size_t)std::max<int64_t>(cur.nnz, 1));
            if (!keys.ptr || !vals.ptr) return NODAL_CUDA_ERROR;
            const int cb = amg_bit_length(nc);
            da_relabel_local_kernel<<<amg_rows_grid(ctx, cur.n), DA, 0, st>>>(cur.n, cur.indptr, cur.indices, cur.data, agg,
                                                                             cur_own, nc, cb, keys, vals);
            KERNEL_CHECK();
            AmgCsr nxt;
            NODAL_TRY(build_rows(S, nc, cur.nnz, cb, keys, vals, 0, nc, &nxt));
            if (cur.owned) amg_free_csr(ctx, cur);
            cur = nxt;
            // global index of the first intermediate row of this rank: the hash must see global edges
            std::vector<int32_t> ib;
            NODAL_TRY(gather_counts(S, nc, ib));
            cur_own = nc;
            cur_base = ib[S.me];
        }
        if (!comp) comp = agg;
        else ctx_pool_free(ctx, agg);
        ncur = nc;
    }
    if (cur.owned) amg_free_csr(ctx, cur);
    NODAL_TRY(gather_counts(S, ncur, *next_bounds));
    const int32_t nc_glob = (*next_bounds)[S.R];
    if ((double)nc_glob > 0.9 * (double)L.nglob) {      // coarsening stalled (same decision on every rank)
        ctx_pool_free(ctx, comp);
        *stalled = true;
        return NODAL_OK;
    }
    // labels of [owned | halo] columns, then the rank's rows of the Galerkin product
    AmgScratch<double> lab(ctx, (size_t)L.halo.ext_len + 2);
    if (!lab.ptr) return NODAL_CUDA_ERROR;
    da_labels_kernel<<<amg_rows_grid(ctx, nloc), DA, 0, st>>>(nloc, comp, (*next_bounds)[S.me], lab);
    KERNEL_CHECK();
    NODAL_TRY(exchange_nccl(S, L.halo, lab, st));
    bool have_members = false;
    if (!S.sorted_galerkin && amg_merge_pays(nnz, ncur)) {
        // members of the composed aggregates (also the restriction pattern), then one thread merges
        // the member rows of its coarse row with the global coarse column ids
        AmgScratch<int32_t> lab32(ctx, (size_t)L.halo.ext_len + 2);
        if (!lab32.ptr) return NODAL_CUDA_ERROR;
        da_labels_to_i32_kernel<<<amg_rows_grid(ctx, L.halo.ext_len), DA, 0, st>>>(L.halo.ext_len, lab, lab32);
        KERNEL_CHECK();
        NODAL_TRY(amg_members(ctx, nloc, comp, ncur, &L.pt_ptr, &L.pt_idx, st));
        S.owned.push_back(L.pt_ptr);
        S.owned.push_back(L.pt_idx);
        have_members = true;
        NODAL_TRY(amg_galerkin_merge(ctx, loc, L.pt_ptr, L.pt_idx, ncur, lab32, 0x7fffffff, next, st));
    } else {
        AmgScratch<u64> keys(ctx, (size_t)std::max<int64_t>(nnz, 1));
        AmgScratch<double> vals(ctx, (size_t)std::max<int64_t>(nnz, 1));
        if (!keys.ptr || !vals.ptr) return NODAL_CUDA_ERROR;
        const int cb = amg_bit_length(nc_glob);
        da_relabel_global_kernel<<<amg_rows_grid(ctx, nloc), DA, 0, st>>>(nloc, L.A.indptr, L.lcols, L.A.data, lab, cb, keys, vals);
        KERNEL_CHECK();
        NODAL_TRY(build_rows(S, nc_glob, nnz, cb, keys, vals, (*next_bounds)[S.me], ncur, next));
    }
    {
        // expander-like graphs fill in instead of shrinking: stop (same decision on every rank;
        // counts in units of 1024 entries keep the all-gathered sums inside int32)
        std::vector<int32_t> fine_k, coarse_k;
        NODAL_TRY(gather_counts(S, (int32_t)(nnz >> 10) + 1, fine_k));
        NODAL_TRY(gather_counts(S, (int32_t)(next->nnz >> 10) + 1, coarse_k));
        S.nnz_k_total += (double)coarse_k[S.R];
        if (S.nnz_k_fine == 0.0) { S.nnz_k_fine = (double)fine_k[S.R]; S.nnz_k_total += S.nnz_k_fine; }
        if ((double)coarse_k[S.R] > S.max_fill * (double)fine_k[S.R] || S.nnz_k_total > S.max_complexity * S.nnz_k_fine) {
            amg_free_csr(ctx, *next);
            ctx_pool_free(ctx, comp);
            *stalled = true;
            return NODAL_OK;
        }
    }
    L.agg = comp;
    S.owned.push_back(comp);
    L.nc = ncur;
    if (!have_members) {
        NODAL_TRY(amg_transpose_pattern(ctx, nloc, comp, &L.pt_ptr, &L.pt_idx, st));
        S.owned.push_back(L.pt_ptr);
        S.owned.push_back(L.pt_idx);
    }
    return NODAL_OK;
}

// All ranks' rows of `A` (partition `bounds`) -> the whole operator on every rank.
int gather_operator(Solver& S, const AmgCsr& A, const std::vector<int32_t>& bounds, AmgCsr* out) {
    nodal_ctx* ctx = S.ctx;
    cudaStream_t st = S.st;
    const int R = S.R, me = S.me;
    if (R == 1) { *out = A; out->owned = false; return NODAL_OK; }
    if (A.nnz >= ((int64_t)1 << 31)) return NODAL_BAD_ARG;
    std::vector<int32_t> nzb;
    NODAL_TRY(gather_counts(S, (int32_t)A.nnz, nzb));
    const int32_t n = bounds[R];
    const int64_t nnz = nzb[R];
    AmgScratch<int32_t> ip(ctx, (size_t)n + 1), ix(ctx, (size_t)std::max<int64_t>(nnz, 1));
    AmgScratch<double> dv(ctx, (size_t)std::max<int64_t>(nnz, 1));
    if (!ip.ptr || !ix.ptr || !dv.ptr) return NODAL_CUDA_ERROR;
    // my pieces in place, then one broadcast per rank and array
    const int32_t nloc = bounds[me + 1] - bounds[me];
    CUDA_TRY(cudaMemcpyAsync(ip.ptr + bounds[me], A.indptr, sizeof(int32_t) * (size_t)nloc, cudaMemcpyDeviceToDevice, st));
    if (A.nnz) {
        CUDA_TRY(cudaMemcpyAsync(ix.ptr + nzb[me], A.indices, sizeof(int32_t) * (size_t)A.nnz, cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(dv.ptr + nzb[me], A.data, sizeof(double) * (size_t)A.nnz, cudaMemcpyDeviceToDevice, st));
    }
    NCCL_TRY(g_nccl.GroupStart());
    for (int o = 0; o < R; ++o) {
        const int32_t rows = bounds[o + 1] - bounds[o], cnt = nzb[o + 1] - nzb[o];
        if (rows) NCCL_TRY(g_nccl.Broadcast(ip.ptr + bounds[o], ip.ptr + bounds[o], rows, ncclInt32, o, S.d->comm, st));
        if (cnt) {
            NCCL_TRY(g_nccl.Broadcast(ix.ptr + nzb[o], ix.ptr + nzb[o], cnt, ncclInt32, o, S.d->comm, st));
            NCCL_TRY(g_nccl.Broadcast(dv.ptr + nzb[o], dv.ptr + nzb[o], cnt, ncclFloat64, o, S.d->comm, st));
        }
    }
    NCCL_TRY(g_nccl.GroupEnd());
    for (int o = 0; o < R; ++o) {
        const int32_t rows = bounds[o + 1] - bounds[o];
        if (rows && nzb[o]) {
            da_offset_indptr_kernel<<<amg_rows_grid(ctx, rows), DA, 0, st>>>(rows, ip.ptr + bounds[o], nzb[o]);
            KERNEL_CHECK();
        }
    }
    da_set_i32_kernel<<<1, 32, 0, st>>>(ip.ptr + n, (int32_t)nnz);
    KERNEL_CHECK();
    out->n = n; out->nnz = nnz; out->owned = true;
    out->indptr = ip.keep(); out->indices = ix.keep(); out->data = dv.keep();
    return NODAL_OK;
}

template <int MODE>
int sweep(Solver& S, const DLevel& L, const double* b, const double* x, double* y, cudaStream_t sx) {
    const nodal_sell* m = L.sell;
    sell_launch(m, [&](auto a) {
        amg_sell_kernel<MODE><<<amg_sell_grid(S.ctx, m->nslices), AT, 0, sx>>>(
            m->n, m->nslices, m->slice_w, a, m->dinv, b, x, S.omega, y, nullptr);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}

// The fused sweeps of the cycle (amg_kernels.cuh), for one rank: the sweeps form x0 and the
// prolongated iterate at every gathered column, which needs them at every column the rank's rows
// touch -- all of them local when there are no halos.
template <int MODE>
int cycle_sweep(Solver& S, const DLevel& L, const double* b, const double* xc, double* y, cudaStream_t sx) {
    const nodal_sell* m = L.sell;
    sell_launch(m, [&](auto a) {
        amg_cycle_sweep_kernel<MODE><<<amg_sell_grid(S.ctx, m->nslices), AT, 0, sx>>>(
            m->n, m->nslices, m->slice_w, a, m->dinv, b, S.omega, L.agg, xc, S.scale, y);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}

// u = M r : one V(1,1) cycle over the distributed levels, the replicated hierarchy below them.
// r: [nloc] of level 0; u: the [owned | halo] vector of level 0 the CG's SpMV gathers from.
// With several ranks x0 and the prolongated iterate are stored and their halos exchanged before
// the sweep that gathers them; with one rank the fused sweeps form them in place.
int cycle(Solver& S, const PcgDev* dev, const double* r0, double* u0, cudaStream_t sx) {
    nodal_ctx* ctx = S.ctx;
    const int ND = (int)S.lv.size() - 1;          // levels 0 .. ND-1 are smoothed here; lv[ND] is gathered
    const bool fused = S.R == 1;
    for (int l = 0; l < ND; ++l) {
        DLevel& L = S.lv[l];
        const double* b = l == 0 ? r0 : L.b;
        if (fused) {
            NODAL_TRY(cycle_sweep<1>(S, L, b, nullptr, L.r, sx));
        } else {
            amg_jacobi0_kernel<<<amg_rows_grid(ctx, L.nloc), AT, 0, sx>>>(L.nloc, L.sell->dinv, b, S.omega, L.x);
            KERNEL_CHECK();
            NODAL_TRY(exchange(S, dev, 2 * l, L.halo, L.x_off, sx));
            NODAL_TRY(sweep<1>(S, L, b, L.x, L.r, sx));
        }
        amg_restrict_kernel<<<amg_rows_grid(ctx, L.nc), AT, 0, sx>>>(L.nc, L.pt_ptr, L.pt_idx, L.r, S.lv[l + 1].b);
        KERNEL_CHECK();
    }
    {
        // first replicated level: all-gather its right-hand side, run the replicated cycle
        DLevel& G = S.lv[ND];
        const double* b = ND == 0 ? r0 : G.b;
        if (S.R == 1) {
            NODAL_TRY(nodal_amg_apply(ctx, S.rep, b, S.xfull, sx));
        } else {
            if (S.p2p) {
                const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(16, ((int64_t)G.nloc * S.R + 4095) / 4096));
                da_exchange_kernel<<<grid, 1024, 0, sx>>>(dev, AMG_SLOTS - 1, S.R, S.me, S.bfull_off, b, nullptr, nullptr,
                                                          S.gather_dest_dev, S.gather_need_dev, S.peer_dev, 1, G.nloc);
                KERNEL_CHECK();
            } else {
                CUDA_TRY(cudaMemcpyAsync(S.gather_stage + (size_t)S.R * S.gmax, b, sizeof(double) * (size_t)G.nloc,
                                         cudaMemcpyDeviceToDevice, sx));
                NCCL_TRY(g_nccl.AllGather(S.gather_stage + (size_t)S.R * S.gmax, S.gather_stage, S.gmax, ncclFloat64,
                                          S.d->comm, sx));
                for (int o = 0; o < S.R; ++o) {
                    const int32_t rows = S.rep_bounds[o + 1] - S.rep_bounds[o];
                    if (rows) CUDA_TRY(cudaMemcpyAsync(S.bfull + S.rep_bounds[o], S.gather_stage + (size_t)o * S.gmax,
                                                       sizeof(double) * (size_t)rows, cudaMemcpyDeviceToDevice, sx));
                }
            }
            NODAL_TRY(nodal_amg_apply(ctx, S.rep, S.bfull, S.xfull, sx));
        }
        if (ND == 0) {
            CUDA_TRY(cudaMemcpyAsync(u0, S.xfull + G.row0, sizeof(double) * (size_t)G.nloc, cudaMemcpyDeviceToDevice, sx));
            return NODAL_OK;
        }
    }
    for (int l = ND - 1; l >= 0; --l) {
        DLevel& L = S.lv[l];
        const double* b = l == 0 ? r0 : L.b;
        const double* xc = (l + 1 == ND) ? S.xfull + S.lv[ND].row0 : S.lv[l + 1].x;
        if (fused) {
            NODAL_TRY(cycle_sweep<2>(S, L, b, xc, l == 0 ? u0 : L.x, sx));
        } else {
            amg_prolong_kernel<<<amg_rows_grid(ctx, L.nloc), AT, 0, sx>>>(L.nloc, L.agg, xc, S.scale, L.x, L.r);
            KERNEL_CHECK();
            NODAL_TRY(exchange(S, dev, 2 * l + 1, L.halo, L.r_off, sx));
            NODAL_TRY(sweep<2>(S, L, b, L.r, l == 0 ? u0 : L.x, sx));
        }
    }
    return NODAL_OK;
}

}  // namespace

extern "C" int nodal_dist_amg_pcg(nodal_ctx* ctx, nodal_dist* d, int32_t n_global, const int32_t* bounds_h,
                                  int64_t nnz, const int32_t* indptr, const int32_t* indices,
                                  const double* data, const double* rhs_local, double* x_local,
                                  const double* params, double rtol, int32_t maxit, int32_t* iters_h,
                                  double* relres_h, double* stats_h, void* stream) {
    NvtxRange nvtx_range("nodal_dist_amg_pcg");
    if (!ctx || !d || !bounds_h || !iters_h || !relres_h) return NODAL_BAD_ARG;
    *iters_h = 0;
    *relres_h = 0.0;
    if (stats_h) memset(stats_h, 0, 32 * sizeof(double));
    CUDA_TRY(cudaSetDevice(ctx->device));
    Solver S;
    S.ctx = ctx; S.d = d; S.R = d->nranks; S.me = d->rank; S.st = (cudaStream_t)stream;
    const int R = S.R, me = S.me;
    cudaStream_t st = S.st;
    const int32_t nloc0 = bounds_h[me + 1] - bounds_h[me];
    if (nloc0 <= 0 || bounds_h[0] != 0 || bounds_h[R] != n_global) {
        nodal_set_error("nodal_dist_amg_pcg: every rank must own at least one row and bounds must span [0, n)");
        return NODAL_BAD_ARG;
    }
    double coarse = 0.0, direct_max = 0.0;
    if (params) {
        if (params[0] >= 1.0) S.passes = (int)params[0];
        coarse = params[1];
        if (params[2] > 0.0) S.omega = params[2];
        if (params[3] > 0.0) S.scale = params[3];
        if (params[4] >= 1.0) S.maxlevels = (int)params[4];
        if (params[5] >= 1.0) S.rounds = (int)params[5];
        direct_max = params[6];
        if (params[7] >= 1.0) S.gather_below = (int64_t)params[7];
        if (params[8] > 0.0) S.max_fill = params[8];
    }
    S.params_rep[0] = S.passes; S.params_rep[1] = coarse; S.params_rep[2] = S.omega; S.params_rep[3] = S.scale;
    S.params_rep[4] = S.maxlevels; S.params_rep[5] = S.rounds; S.params_rep[6] = direct_max;
    S.params_rep[7] = S.max_fill;

    cudaEvent_t ev0, ev1, ev2, ev_poll[2];
    CUDA_TRY(cudaEventCreate(&ev0));
    CUDA_TRY(cudaEventCreate(&ev1));
    CUDA_TRY(cudaEventCreate(&ev2));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[0], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[1], cudaEventDisableTiming));
    cudaGraph_t graph[2] = {nullptr, nullptr};
    cudaGraphExec_t gexec[2] = {nullptr, nullptr};
    cudaStream_t cap = nullptr;
    PcgDev host{};
    int restarts = 0;
    float ms_setup = 0.f, ms_solve = 0.f;
    double relres = 0.0;
    unsigned long long launches_per_iter = 0;
    char* local_buf = nullptr;

    auto run = [&]() -> int {
        CUDA_TRY(cudaEventRecord(ev0, st));
        std::unique_ptr<NvtxRange> phase(new NvtxRange("amg setup (hierarchy, halo plans, buffers)"));
        // ---------------- level 0 and the distributed coarsening ----------------
        {
            DLevel L;
            L.bounds.assign(bounds_h, bounds_h + R + 1);
            L.nloc = nloc0; L.row0 = bounds_h[me]; L.nglob = n_global;
            L.A.n = nloc0; L.A.nnz = nnz; L.A.indptr = indptr; L.A.indices = indices; L.A.data = data; L.A.owned = false;
            S.lv.push_back(L);
        }
        for (;;) {
            DLevel& L = S.lv.back();
            const bool fine = S.lv.size() == 1;
            const bool distribute = (int64_t)L.nglob > S.gather_below && (int)S.lv.size() < S.maxlevels;
            if (fine || distribute) {
                NODAL_TRY(build_halo(S, L));
                NODAL_TRY(sell_from_csr(ctx, L.nloc, L.A.nnz, L.A.indptr, L.lcols, L.A.data, &L.sell, st, nullptr));
            }
            if (!distribute) break;
            AmgCsr next;
            std::vector<int32_t> nb;
            bool stalled = false;
            NODAL_TRY(coarsen(S, L, &next, &nb, &stalled));
            if (stalled) break;
            DLevel C;
            C.bounds = nb;
            C.nloc = nb[me + 1] - nb[me]; C.row0 = nb[me]; C.nglob = nb[R];
            C.A = next;
            S.lv.push_back(C);      // (invalidates L)
        }
        const int ND = (int)S.lv.size() - 1;
        if (ND == 0 && (int64_t)S.lv[0].nglob > S.gather_below) {
            // the finest level did not coarsen (stalled: hardly fewer rows or entries): replicating
            // it on every rank would make every rank do the whole job.  Same decision everywhere.
            nodal_set_error("nodal_dist_amg_pcg: the aggregation hierarchy stalled on the finest level "
                            "(expander-like graph); use the Jacobi-preconditioned solver");
            return NODAL_BREAKDOWN;
        }
        if (2 * ND + 2 > AMG_SLOTS - 1) { nodal_set_error("nodal_dist_amg_pcg: too many distributed levels"); return NODAL_BAD_ARG; }
        // ---------------- replicated hierarchy below ----------------
        {
            DLevel& G = S.lv[ND];
            S.rep_bounds = G.bounds;
            S.rep_n = G.nglob;
            NODAL_TRY(gather_operator(S, G.A, G.bounds, &S.repA));
            NODAL_TRY(nodal_amg_create(ctx, S.repA.n, S.repA.nnz, S.repA.indptr, S.repA.indices, S.repA.data,
                                       S.params_rep, &S.rep, st));
            for (int o = 0; o < R; ++o) S.gmax = std::max(S.gmax, G.bounds[o + 1] - G.bounds[o]);
        }
        // ---------------- exchange buffer: mailbox + every [owned | halo] vector ----------------
        size_t bytes = AMG_HDR;
        auto place = [&](int64_t doubles) { const long long off = (long long)bytes; bytes += align_up((size_t)doubles * 8, 256); return off; };
        const long long u_off = place(S.lv[0].slot_len);
        const long long xs_off = place(S.lv[0].slot_len);     // x in the [owned | halo] layout (true residuals)
        for (int l = 0; l < ND; ++l) { S.lv[l].x_off = place(S.lv[l].slot_len); S.lv[l].r_off = place(S.lv[l].slot_len); }
        S.bfull_off = place((int64_t)S.rep_n + 2);
        bool usable = false;
        NODAL_TRY(peer_heap_ensure(ctx, d, &d->amg, bytes, AMG_HDR, st, &usable));
        S.p2p = usable;
        if (S.p2p) {
            S.base = d->amg.shm;
            S.peer_dev = d->amg.peer_dev;
        } else {
            local_buf = static_cast<char*>(ctx_pool_alloc(ctx, bytes));
            if (!local_buf) return NODAL_CUDA_ERROR;
            CUDA_TRY(cudaMemsetAsync(local_buf, 0, AMG_HDR, st));
            S.base = local_buf;
        }
        double* u = reinterpret_cast<double*>(S.base + u_off);
        for (int l = 0; l < ND; ++l) {
            DLevel& L = S.lv[l];
            L.x = reinterpret_cast<double*>(S.base + L.x_off);
            L.r = reinterpret_cast<double*>(S.base + L.r_off);
        }
        for (int l = 1; l <= ND; ++l) {
            S.lv[l].b = S.alloc<double>((size_t)S.lv[l].nloc + 2);
            if (!S.lv[l].b) return NODAL_CUDA_ERROR;
        }
        S.bfull = reinterpret_cast<double*>(S.base + S.bfull_off);
        S.xfull = S.alloc<double>((size_t)S.rep_n + 2);
        if (!S.xfull) return NODAL_CUDA_ERROR;
        if (R > 1) {
            std::vector<long long> gd(R, (long long)S.rep_bounds[me]);
            std::vector<int32_t> gn(R);
            for (int o = 0; o < R; ++o) gn[o] = S.rep_bounds[o + 1] - S.rep_bounds[o];
            S.gather_dest_dev = S.alloc<long long>((size_t)R);
            S.gather_need_dev = S.alloc<int32_t>((size_t)R);
            S.gather_stage = S.alloc<double>((size_t)(R + 1) * S.gmax + 2);
            if (!S.gather_dest_dev || !S.gather_need_dev || !S.gather_stage) return NODAL_CUDA_ERROR;
            CUDA_TRY(cudaMemcpyAsync(S.gather_dest_dev, gd.data(), sizeof(long long) * (size_t)R, cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(S.gather_need_dev, gn.data(), sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        // ---------------- CG vectors ----------------
        DLevel& F = S.lv[0];
        const int32_t n = F.nloc;
        const int gv = amg_rows_grid(ctx, n);
        const int gs = amg_sell_grid(ctx, F.sell->nslices);
        const int gmaxp = std::max(gv, gs) + 1;
        double* r = S.alloc<double>((size_t)n + 2);
        double* p = S.alloc<double>((size_t)n + 2);
        double* s = S.alloc<double>((size_t)n + 2);
        double* w = S.alloc<double>((size_t)n + 2);
        double* part = S.alloc<double>(4 * (size_t)gmaxp + 64);
        PcgDev* dev = S.alloc<PcgDev>(1);
        if (!r || !p || !s || !w || !part || !dev) return NODAL_CUDA_ERROR;
        double* part_g = part;
        double* part_d = part + gmaxp;
        double* part_rr = part + 2 * (size_t)gmaxp;
        double* part_bb = part + 3 * (size_t)gmaxp;
        double* SC = part + 4 * (size_t)gmaxp;                   // SC[par * 4 + {gamma, delta, rr, alpha}], [12..15] scratch
        CUDA_TRY(cudaMemsetAsync(dev, 0, sizeof(PcgDev), st));
        CUDA_TRY(cudaMemsetAsync(SC, 0, sizeof(double) * 32, st));
        const int use_mail = (S.p2p && R > 1) ? 1 : 0;

        auto allreduce = [&](int check_done, const double* a, int na, const double* b, int nb, const double* c, int nc,
                             const double* dd, int nd, double* out, int enforce, cudaStream_t sx) -> int {
            acg_allreduce_kernel<<<1, DA, 0, sx>>>(dev, check_done, a, na, b, nb, c, nc, dd, nd, R, me, S.peer_dev, use_mail,
                                                   out, enforce);
            KERNEL_CHECK();
            if (R > 1 && !use_mail) NCCL_TRY(g_nccl.AllReduce(out, out, 4, ncclFloat64, ncclSum, d->comm, sx));
            return NODAL_OK;
        };
        // (re)start from the current x: r = b - A x, u = M r, w = A u, p = s = 0.  x is staged in its
        // own [owned | halo] vector and slot: no buffer is written twice between two all-reduces.
        double* xstage = reinterpret_cast<double*>(S.base + xs_off);
        auto start = [&](int first) -> int {
            CUDA_TRY(cudaMemcpyAsync(xstage, x_local, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, st));
            NODAL_TRY(exchange(S, nullptr, AMG_SLOTS - 2, F.halo, xs_off, st));
            NODAL_TRY(sweep<1>(S, F, rhs_local, xstage, r, st));          // r = b - A x
            acg_start_kernel<<<gv, DA, 0, st>>>(n, rhs_local, r, p, s, part_rr, part_bb);
            KERNEL_CHECK();
            NODAL_TRY(cycle(S, nullptr, r, u, st));
            NODAL_TRY(exchange(S, nullptr, 2 * ND, F.halo, u_off, st));
            sell_launch(F.sell, [&](auto a) {
                acg_spmv_dots_kernel<<<gs, DA, 0, st>>>(n, F.sell->nslices, F.sell->slice_w, a, u, r, w, part_g, part_d);
            });
            KERNEL_CHECK();
            NODAL_TRY(allreduce(0, part_g, gs, part_d, gs, part_rr, gv, part_bb, gv, SC, 0, st));
            acg_scalars_kernel<<<1, 32, 0, st>>>(dev, SC, rtol, maxit, first);
            KERNEL_CHECK();
            return NODAL_OK;
        };
        auto iteration = [&](int par, cudaStream_t sx) -> int {
            double* cur = SC + par * 4;
            double* nxt = SC + (par ^ 1) * 4;
            acg_vector_kernel<<<gv, DA, 0, sx>>>(dev, n, cur, nxt, x_local, r, p, s, u, w, part_rr);
            KERNEL_CHECK();
            NODAL_TRY(cycle(S, dev, r, u, sx));
            NODAL_TRY(exchange(S, dev, 2 * ND, F.halo, u_off, sx));
            sell_launch(F.sell, [&](auto a) {
                acg_spmv_dots_kernel<<<gs, DA, 0, sx>>>(n, F.sell->nslices, F.sell->slice_w, a, u, r, w, part_g, part_d);
            });
            KERNEL_CHECK();
            NODAL_TRY(allreduce(1, part_g, gs, part_d, gs, part_rr, gv, nullptr, 0, nxt, 1, sx));
            return NODAL_OK;
        };
        nvtxRangePushA("amg first residual + cycle");
        const int start_rc = start(1);
        nvtxRangePop();
        NODAL_TRY(start_rc);
        const bool use_graph = getenv("NODAL_DIST_NO_GRAPH") == nullptr;
        if (use_graph) {
            const unsigned long long before = g_nodal_launches;
            CUDA_TRY(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
            for (int par = 0; par < 2; ++par) {
                CUDA_TRY(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
                const int crc = iteration(par, cap);
                cudaError_t ce = cudaStreamEndCapture(cap, &graph[par]);
                if (crc != NODAL_OK) return crc;
                CUDA_TRY(ce);
                CUDA_TRY(cudaGraphInstantiate(&gexec[par], graph[par], 0));
            }
            launches_per_iter = (g_nodal_launches - before) / 2;
            g_nodal_launches = before;
        }
        CUDA_TRY(cudaEventRecord(ev1, st));
        phase.reset();
        phase.reset(new NvtxRange("amg-pcg iterations"));
        PcgDev* poll = reinterpret_cast<PcgDev*>(ctx->pinned);
        double last_true_rr = -1.0;
        int par = 0;
        for (;;) {
            int64_t k = 0;
            const int64_t max_iters = (int64_t)maxit + 4;
            for (;; ++k) {
                if (use_graph) {
                    CUDA_TRY(cudaGraphLaunch(gexec[par], st));
                    g_nodal_launches += launches_per_iter;
                } else {
                    NODAL_TRY(iteration(par, st));
                }
                par ^= 1;
                CUDA_TRY(cudaMemcpyAsync(&poll[k & 1], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaEventRecord(ev_poll[k & 1], st));
                if (R > 1 && !use_mail) {
                    // NCCL back end: the collectives inside an iteration do not look at the `done` word,
                    // so every rank must launch exactly the same number of iterations: no look-ahead
                    CUDA_TRY(cudaEventSynchronize(ev_poll[k & 1]));
                    if (poll[k & 1].done) break;
                    if (k > max_iters) break;
                    continue;
                }
                if (k >= 1) {
                    CUDA_TRY(cudaEventSynchronize(ev_poll[(k - 1) & 1]));
                    if (poll[(k - 1) & 1].done) break;
                }
                if (k > max_iters) break;
            }
            CUDA_TRY(cudaStreamSynchronize(st));
            host = poll[k & 1];
            if (!host.done) host.status = NODAL_NOT_CONVERGED;
            if (host.status == NODAL_BREAKDOWN || host.status == NODAL_CUDA_ERROR) break;
            const int recurrence_status = host.status;
            const int iters_so_far = host.iters;
            NODAL_TRY(start(0));     // true residual of the current x (and a restart, if needed)
            par = 0;
            CUDA_TRY(cudaMemcpyAsync(&poll[0], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            host = poll[0];
            host.iters = iters_so_far;
            if (host.rr <= host.tol2) { host.status = NODAL_OK; break; }
            if (!(host.rr == host.rr)) { host.status = NODAL_BREAKDOWN; break; }
            if (recurrence_status == NODAL_NOT_CONVERGED || host.iters >= host.maxit) { host.status = NODAL_NOT_CONVERGED; break; }
            if (restarts >= 8 || (last_true_rr >= 0.0 && host.rr > 0.25 * last_true_rr)) { host.status = NODAL_NOT_CONVERGED; break; }
            last_true_rr = host.rr;
            ++restarts;
        }
        CUDA_TRY(cudaEventRecord(ev2, st));
        CUDA_TRY(cudaEventSynchronize(ev2));
        CUDA_TRY(cudaEventElapsedTime(&ms_setup, ev0, ev1));
        CUDA_TRY(cudaEventElapsedTime(&ms_solve, ev1, ev2));
        relres = host.bb > 0.0 ? sqrt(host.rr / host.bb) : 0.0;
        if (S.p2p) {
            unsigned long long err = 0;
            CUDA_TRY(cudaMemcpy(&err, &reinterpret_cast<AmgMail*>(S.base)->err, sizeof(err), cudaMemcpyDeviceToHost));
            if (err) {
                nodal_set_error("nodal_dist_amg_pcg: a peer-memory exchange timed out (rank %d)", me);
                CUDA_TRY(cudaMemset(&reinterpret_cast<AmgMail*>(S.base)->err, 0, sizeof(err)));
                return NODAL_CUDA_ERROR;
            }
        }
        return host.status;
    };
    const int rc = run();
    cudaStreamSynchronize(st);
    // ---------------- statistics and teardown ----------------
    *iters_h = host.iters;
    *relres_h = relres;
    if (stats_h) {
        int32_t nl = 0;
        int64_t rows[64], nnzs[64];
        double rep_ms = 0.0;
        int32_t direct = 0;
        if (S.rep) nodal_amg_info(S.rep, 64, &nl, rows, nnzs, &rep_ms, &direct);
        stats_h[0] = (double)((int)S.lv.size() - 1 + nl);      // levels: distributed + replicated
        stats_h[2] = restarts;
        stats_h[3] = ms_solve;
        stats_h[4] = ms_setup;
        stats_h[5] = nl > 0 ? (double)rows[nl - 1] : 0.0;
        stats_h[7] = direct;
        stats_h[8] = (double)((int)S.lv.size() - 1);            // distributed levels
        stats_h[9] = S.p2p ? 2.0 : 0.0;
        stats_h[10] = (double)launches_per_iter;
        stats_h[11] = (double)S.rep_n;
        stats_h[12] = (double)S.halo_total;
        for (size_t l = 0; l < S.lv.size() && l < 12; ++l) stats_h[16 + l] = (double)S.lv[l].nglob;
    }
    for (int par = 0; par < 2; ++par) {
        if (gexec[par]) cudaGraphExecDestroy(gexec[par]);
        if (graph[par]) cudaGraphDestroy(graph[par]);
    }
    if (cap) cudaStreamDestroy(cap);
    if (S.rep) nodal_amg_destroy(S.rep);
    if (S.repA.owned) amg_free_csr(ctx, S.repA);
    for (size_t l = 0; l < S.lv.size(); ++l) {
        if (S.lv[l].sell) sell_free(S.lv[l].sell);
        if (l > 0 && S.lv[l].A.owned) amg_free_csr(ctx, S.lv[l].A);
    }
    for (void* ptr : S.owned) ctx_pool_free(ctx, ptr);
    if (local_buf) ctx_pool_free(ctx, local_buf);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1); cudaEventDestroy(ev2);
    cudaEventDestroy(ev_poll[0]); cudaEventDestroy(ev_poll[1]);
    return rc;
}
