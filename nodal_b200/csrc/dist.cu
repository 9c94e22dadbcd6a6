// Row-partitioned Jacobi-PCG across GPUs (one process per GPU), NCCL over NVLink/NVSwitch.
//
// Rank k owns the contiguous rows [bounds[k], bounds[k+1]) of G as a local CSR with GLOBAL
// column indices.  Setup (all on device except the tiny per-peer bookkeeping):
//   - the off-rank columns referenced by local rows are compacted, radix-sorted and made
//     unique -> the halo list; columns are renumbered to the local layout
//     [ owned x (nloc) | halo x (nhalo) ];
//   - ranks tell every owner which entries they need (ncclAllGather of the count matrix,
//     grouped ncclSend/ncclRecv of the index lists).
// Iteration (Chronopoulos-Gear single-reduction form of Jacobi-PCG, see cgcg_vector_kernel):
//   - one fused vector kernel (p, s, x, r, u updates + partial dots),
//   - gather of the entries peers need + grouped ncclSend/ncclRecv straight into the halo
//     tail of u,
//   - the single-GPU SpMV+dot kernel (pcg_kernels.cuh) on the local rows,
//   - ONE ncclAllReduce of 3 doubles (r.u, w.u, r.r).
// A chunk of 32 iterations, NCCL calls included, is captured in one CUDA graph.
// The scalar results are bitwise identical on all ranks, so every rank takes the same
// convergence decision with no extra traffic.  libnccl.so.2 is dlopen'ed: the single-GPU
// library has no NCCL dependency.
#include <algorithm>
#include <chrono>
#include <vector>

#include "dist_common.cuh"
#include "pcg_kernels.cuh"

NcclApi g_nccl;

int load_nccl() {
    if (g_nccl.handle) return NODAL_OK;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
        nodal_set_error("cannot dlopen libnccl.so.2: %s", dlerror());
        return NODAL_CUDA_ERROR;
    }
#define SYM(field, name)                                                      \
    g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(h, name)); \
    if (!g_nccl.field) {                                                      \
        nodal_set_error("libnccl: missing symbol %s", name);                  \
        return NODAL_CUDA_ERROR;                                              \
    }
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(AllReduce, "ncclAllReduce")
    SYM(AllGather, "ncclAllGather")
    SYM(Broadcast, "ncclBroadcast")
    SYM(Send, "ncclSend")
    SYM(Recv, "ncclRecv")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    g_nccl.handle = h;
    return NODAL_OK;
}

// The PCG's peer-mapped buffer: a 4 KB mailbox followed by the rank's u vector [owned | halo].
constexpr size_t P2P_HDR = 4096;
struct P2PMail {
    double red[2][P2P_MAXR][4];            // [parity][source rank] = {gamma, delta, rr, tag}
    unsigned long long hflag[P2P_MAXR];    // halo of iteration `tag` from that rank has landed
    unsigned long long err;
};

void peer_heap_release(nodal_dist* d, PeerHeap* h) {
    for (size_t o = 0; o < h->peer.size(); ++o)
        if ((int)o != d->rank && h->peer[o]) cudaIpcCloseMemHandle(h->peer[o]);
    h->peer.clear();
    if (h->shm) cudaFree(h->shm);
    if (h->peer_dev) cudaFree(h->peer_dev);
    if (h->seq) cudaFree(h->seq);
    h->shm = nullptr; h->peer_dev = nullptr; h->seq = nullptr; h->bytes = 0;
}

extern "C" int nodal_dist_unique_id(uint8_t* id_h) {
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    NODAL_TRY(load_nccl());
    ncclUniqueId id;
    NCCL_TRY(g_nccl.GetUniqueId(&id));
    memcpy(id_h, &id, sizeof(id));
    return NODAL_OK;
}

extern "C" int nodal_dist_create(nodal_ctx* ctx, const uint8_t* id_h, int32_t rank, int32_t nranks,
                                 nodal_dist** out) {
    if (!ctx || !id_h || !out || rank < 0 || rank >= nranks) return NODAL_BAD_ARG;
    NODAL_TRY(load_nccl());
    CUDA_TRY(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id_h, sizeof(id));
    nodal_dist* d = new nodal_dist();
    d->rank = rank;
    d->nranks = nranks;
    d->device = ctx->device;
    ncclResult_t r = g_nccl.CommInitRank(&d->comm, nranks, id, rank);
    if (r != ncclSuccess) {
        nodal_set_error("ncclCommInitRank -> %s", g_nccl.GetErrorString(r));
        delete d;
        return NODAL_CUDA_ERROR;
    }
    *out = d;
    return NODAL_OK;
}

// A one-rank object without a communicator (no NCCL needed): the row-partitioned drivers run
// with empty halos, which makes nodal_dist_amg_pcg the graph-captured single-GPU AMG-PCG.
extern "C" int nodal_dist_create_single(nodal_ctx* ctx, nodal_dist** out) {
    if (!ctx || !out) return NODAL_BAD_ARG;
    nodal_dist* d = new nodal_dist();
    d->rank = 0;
    d->nranks = 1;
    d->device = ctx->device;
    *out = d;
    return NODAL_OK;
}

extern "C" int nodal_dist_destroy(nodal_dist* d) {
    if (!d) return NODAL_OK;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    peer_heap_release(d, &d->pcg);
    peer_heap_release(d, &d->amg);
    if (d->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(d->comm);
    delete d;
    return NODAL_OK;
}

// ---------------------------------------------------------------- setup kernels
constexpr int DT = 256;

__global__ void __launch_bounds__(DT)
dist_flag_external_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re,
                          u32* __restrict__ flag) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t c = cols[i];
        flag[i] = (c < rb || c >= re) ? 1u : 0u;
    }
}

__global__ void __launch_bounds__(DT)
dist_compact_external_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re,
                             const u32* __restrict__ pos, u64* __restrict__ keys) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t c = cols[i];
        if (c < rb || c >= re) keys[pos[i]] = (u64)(u32)c;
    }
}

__global__ void __launch_bounds__(DT)
dist_unique_flag_kernel(int64_t m, const u64* __restrict__ keys, u32* __restrict__ flag) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        flag[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(DT)
dist_unique_compact_kernel(int64_t m, const u64* __restrict__ keys, const u32* __restrict__ pos,
                           int32_t* __restrict__ halo) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        if (i == 0 || keys[i] != keys[i - 1]) halo[pos[i]] = (int32_t)keys[i];
}

// global column -> local layout [owned | halo]
__global__ void __launch_bounds__(DT)
dist_remap_kernel(int64_t nnz, const int32_t* __restrict__ cols, int32_t rb, int32_t re,
                  const int32_t* __restrict__ halo, int32_t nhalo, int32_t* __restrict__ out) {
    const int32_t nloc = re - rb;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
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

__global__ void __launch_bounds__(DT)
dist_rebase_kernel(int64_t m, int32_t* __restrict__ idx, int32_t rb) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        idx[i] -= rb;
}

__global__ void __launch_bounds__(DT)
dist_gather_kernel(int64_t m, const int32_t* __restrict__ idx, const double* __restrict__ src,
                   double* __restrict__ dst) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[idx[i]];
}

// out[k] = deterministic sum of partial array k (up to 3 arrays)
__global__ void __launch_bounds__(PCG_THREADS)
dist_reduce_kernel(const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c,
                   int count, double* __restrict__ out) {
    __shared__ double sm[40];
    const double sa = reduce_partials(a, count, sm);
    const double sb = b ? reduce_partials(b, count, sm) : 0.0;
    const double sc = c ? reduce_partials(c, count, sm) : 0.0;
    if (threadIdx.x == 0) {
        out[0] = sa;
        if (b) out[1] = sb;
        if (c) out[2] = sc;
    }
}

// ---------------------------------------------------------------- single-reduction CG kernels
// Chronopoulos-Gear form of Jacobi-PCG: one fused vector pass + one SpMV per iteration and a
// single all-reduce of (gamma, delta, rr):
//   beta = gamma_i / gamma_{i-1} ; alpha = gamma_i / (delta_i - beta gamma_i / alpha_{i-1})
//   p = u + beta p ; s = w + beta s ; x += alpha p ; r -= alpha s ; u = D^-1 r
//   w = A u ; gamma_{i+1} = r.u ; delta_{i+1} = w.u ; rr = r.r
// SC holds two parity slots {gamma, delta, rr, alpha}; alpha == 0 in the previous slot marks the
// first iteration after a (re)start.
template <bool UNIT>
__global__ void __launch_bounds__(PCG_THREADS)
cgcg_vector_kernel(PcgDev* __restrict__ dev, int32_t n, double* __restrict__ cur, const double* __restrict__ prev,
                   double* __restrict__ x, double* __restrict__ r, double* __restrict__ p,
                   double* __restrict__ s, const double* __restrict__ w, const double* __restrict__ dinv,
                   double* __restrict__ u, double* __restrict__ part_g, double* __restrict__ part_rr) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    const double g = cur[0], dl = cur[1], rr = cur[2];
    const double gp = prev[0], ap = prev[3];
    const bool conv = rr <= dev->tol2;
    double beta = 0.0, den = dl;
    if (ap != 0.0) { beta = g / gp; den = dl - beta * g / ap; }
    const double alpha = g / den;
    const bool bad = !(den > 0.0) || !(rr == rr);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        dev->rr = rr;
        if (conv) { dev->done = 1; dev->status = NODAL_OK; }
        else if (bad) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
        else { dev->iters = dev->iters + 1; cur[3] = alpha; }
    }
    if (conv || bad) return;
    double lg = 0.0, lrr = 0.0;
    const int64_t n2 = n >> 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    double2* x2 = reinterpret_cast<double2*>(x);
    double2* r2 = reinterpret_cast<double2*>(r);
    double2* p2 = reinterpret_cast<double2*>(p);
    double2* s2 = reinterpret_cast<double2*>(s);
    double2* u2 = reinterpret_cast<double2*>(u);
    const double2* w2 = reinterpret_cast<const double2*>(w);
    const double2* d2 = reinterpret_cast<const double2*>(dinv);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
        double2 xv = x2[i], rv = r2[i], pv = p2[i], sv = s2[i];
        const double2 wv = w2[i];
        double2 dv = make_double2(1.0, 1.0);
        if (!UNIT) dv = d2[i];
        pv.x = fma(beta, pv.x, dv.x * rv.x); pv.y = fma(beta, pv.y, dv.y * rv.y);
        sv.x = fma(beta, sv.x, wv.x);        sv.y = fma(beta, sv.y, wv.y);
        xv.x = fma(alpha, pv.x, xv.x);       xv.y = fma(alpha, pv.y, xv.y);
        rv.x = fma(-alpha, sv.x, rv.x);      rv.y = fma(-alpha, sv.y, rv.y);
        p2[i] = pv; s2[i] = sv; x2[i] = xv; r2[i] = rv;
        if (!UNIT) {
            double2 uv;
            uv.x = dv.x * rv.x; uv.y = dv.y * rv.y;
            u2[i] = uv;
            lg = fma(rv.x, uv.x, lg); lg = fma(rv.y, uv.y, lg);
        }
        lrr = fma(rv.x, rv.x, lrr); lrr = fma(rv.y, rv.y, lrr);
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t i = n - 1;
        const double dvi = UNIT ? 1.0 : dinv[i];
        const double pv = fma(beta, p[i], dvi * r[i]);
        const double sv = fma(beta, s[i], w[i]);
        const double rv = fma(-alpha, sv, r[i]);
        p[i] = pv; s[i] = sv; x[i] = fma(alpha, pv, x[i]); r[i] = rv;
        if (!UNIT) { const double uv = dvi * rv; u[i] = uv; lg = fma(rv, uv, lg); }
        lrr = fma(rv, rv, lrr);
    }
    lrr = block_sum(lrr, sm);
    lg = UNIT ? lrr : block_sum(lg, sm);
    if (threadIdx.x == 0) { part_g[blockIdx.x] = lg; part_rr[blockIdx.x] = lrr; }
}

// r = b - q ; u = D^-1 r ; p = s = 0 ; partial sums of r.u, r.r, b.b
template <bool UNIT>
__global__ void __launch_bounds__(PCG_THREADS)
cgcg_start_kernel(int32_t n, const double* __restrict__ b, const double* __restrict__ q,
                  const double* __restrict__ dinv, double* __restrict__ r, double* __restrict__ u,
                  double* __restrict__ p, double* __restrict__ s, double* __restrict__ part_g,
                  double* __restrict__ part_rr, double* __restrict__ part_bb) {
    __shared__ double sm[40];
    double lg = 0.0, lrr = 0.0, lbb = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double bv = b[i];
        const double rv = bv - q[i];
        const double uv = UNIT ? rv : rv * dinv[i];
        r[i] = rv; p[i] = 0.0; s[i] = 0.0;
        if (!UNIT) u[i] = uv;
        lg = fma(rv, uv, lg);
        lrr = fma(rv, rv, lrr);
        lbb = fma(bv, bv, lbb);
    }
    lg = block_sum(lg, sm);
    lrr = block_sum(lrr, sm);
    lbb = block_sum(lbb, sm);
    if (threadIdx.x == 0) { part_g[blockIdx.x] = lg; part_rr[blockIdx.x] = lrr; part_bb[blockIdx.x] = lbb; }
}

__global__ void cgcg_reset_kernel(PcgDev* dev) {
    if (threadIdx.x == 0) dev->done = 0;
}

// out = {sum part_g, sum part_d, sum part_rr [, sum part_bb]} ; also enforces maxit
__global__ void __launch_bounds__(PCG_THREADS)
cgcg_reduce_kernel(PcgDev* __restrict__ dev, const double* __restrict__ part_g, const double* __restrict__ part_rr,
                   const double* __restrict__ part_bb, int cnt_v, const double* __restrict__ part_d, int cnt_s,
                   double* __restrict__ out, int with_bb) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    const double g = reduce_partials(part_g, cnt_v, sm);
    const double rr = reduce_partials(part_rr, cnt_v, sm);
    const double dl = reduce_partials(part_d, cnt_s, sm);
    const double bb = with_bb ? reduce_partials(part_bb, cnt_v, sm) : 0.0;
    if (threadIdx.x == 0) {
        out[0] = g; out[1] = dl; out[2] = rr;
        if (with_bb) out[3] = bb;
        else if (dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
    }
}

// after the start all-reduce: SC[0..3] = {gamma, delta, rr, bb}
__global__ void cgcg_scalars_kernel(PcgDev* dev, double* SC, double rtol, int maxit, int first) {
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

// ---------------------------------------------------------------- peer-memory kernels
// One CTA: copy the entries every peer needs from my u into the halo tail of THEIR u, then
// raise my flag in their mailbox.
__global__ void __launch_bounds__(1024)
p2p_push_kernel(const PcgDev* __restrict__ dev, const unsigned long long* __restrict__ seq, int R, int me,
                const int32_t* __restrict__ send_idx, const int32_t* __restrict__ send_off,
                const long long* __restrict__ dest_off, char* const* __restrict__ peer,
                const double* __restrict__ u) {
    if (block_done(&dev->done)) return;
    const unsigned long long tag = *seq + 1;
    for (int o = 0; o < R; ++o) {
        if (o == me) continue;
        const int b = send_off[o], e = send_off[o + 1];
        double* dst = reinterpret_cast<double*>(peer[o] + P2P_HDR) + dest_off[o];
        for (int j = b + threadIdx.x; j < e; j += blockDim.x) dst[j - b] = u[send_idx[j]];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < R && threadIdx.x != me && send_off[threadIdx.x + 1] > send_off[threadIdx.x]) {
        P2PMail* m = reinterpret_cast<P2PMail*>(peer[threadIdx.x]);
        __threadfence_system();
        st_sys_u64(&m->hflag[me], tag);
    }
}

// One warp: wait until every neighbour's halo block of this iteration has landed in my u.
__global__ void p2p_wait_halo_kernel(PcgDev* __restrict__ dev, const unsigned long long* __restrict__ seq, int R,
                                     int me, const int32_t* __restrict__ need_cnt, P2PMail* mine) {
    if (*reinterpret_cast<volatile int*>(&dev->done)) return;
    const unsigned long long tag = *seq + 1;
    const int o = threadIdx.x;
    bool timeout = false;
    if (o < R && o != me && need_cnt[o] > 0) {
        const long long t0 = clock64();
        while (ld_sys_u64(&mine->hflag[o]) < tag) {
            if (clock64() - t0 > P2P_SPIN_LIMIT) { timeout = true; break; }
        }
    }
    if (__any_sync(0xffffffffu, timeout) && threadIdx.x == 0) {
        dev->done = 1;
        dev->status = NODAL_CUDA_ERROR;
        mine->err = 1;
    }
    __threadfence_system();
}

// One CTA: local sums -> every rank's mailbox; wait for all ranks; sum in rank order (the
// result is bitwise identical everywhere); advance the sequence number.
__global__ void __launch_bounds__(PCG_THREADS)
p2p_reduce_kernel(PcgDev* __restrict__ dev, unsigned long long* __restrict__ seq, int R, int me,
                  const double* __restrict__ part_g, const double* __restrict__ part_rr, int cnt_v,
                  const double* __restrict__ part_d, int cnt_s, char* const* __restrict__ peer,
                  double* __restrict__ out) {
    __shared__ double sm[40];
    __shared__ int s_timeout;
    if (block_done(&dev->done)) return;
    const double g = reduce_partials(part_g, cnt_v, sm);
    const double rr = reduce_partials(part_rr, cnt_v, sm);
    const double dl = reduce_partials(part_d, cnt_s, sm);
    const unsigned long long s0 = *seq;
    const unsigned long long tag = s0 + 1;
    const int par = (int)(s0 & 1ull);
    if (threadIdx.x == 0) s_timeout = 0;
    __syncthreads();
    if (threadIdx.x < R) {
        P2PMail* m = reinterpret_cast<P2PMail*>(peer[threadIdx.x]);
        volatile double* slot = m->red[par][me];
        slot[0] = g; slot[1] = dl; slot[2] = rr;
        __threadfence_system();
        st_sys_u64(reinterpret_cast<unsigned long long*>(&m->red[par][me][3]), tag);
    }
    P2PMail* mine = reinterpret_cast<P2PMail*>(peer[me]);
    if (threadIdx.x < R) {
        const unsigned long long* tp = reinterpret_cast<const unsigned long long*>(&mine->red[par][threadIdx.x][3]);
        const long long t0 = clock64();
        while (ld_sys_u64(tp) != tag) {
            if (clock64() - t0 > P2P_SPIN_LIMIT) { s_timeout = 1; break; }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_timeout) {
            dev->done = 1; dev->status = NODAL_CUDA_ERROR; mine->err = 1;
        } else {
            double sg = 0.0, sd = 0.0, sr = 0.0;
            for (int t = 0; t < R; ++t) {
                const volatile double* slot = mine->red[par][t];
                sg += slot[0]; sd += slot[1]; sr += slot[2];
            }
            out[0] = sg; out[1] = sd; out[2] = sr;
            *seq = tag;
            if (dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        }
    }
}

// ---------------------------------------------------------------- fused peer-memory iteration
// Two kernels per iteration.  The vector pass ends with the halo push (done by whichever CTA
// finishes last); the SpMV starts by waiting for the neighbours' pushes and ends with the
// mailbox all-reduce (again the last CTA).  Reduction order is fixed, so the result does not
// depend on which CTA happens to be last.
struct DistSync {
    unsigned int ticket_v[64], ticket_s[64];   // [0] = top level, [1 + g] = group g of 32 CTAs
    unsigned long long dbg[16];                // ns accumulated in the tails (diagnostics)
};
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// "Am I the last CTA of the grid to get here?"  Two-level ticket so that no address sees more
// than ~37 arrivals (a single counter serialises ~1200 same-address atomics, 10+ us).
__device__ __forceinline__ bool last_cta_arrive(unsigned int* tickets, int* s_flag) {
    __syncthreads();          // the CTA's writes are ordered before thread 0 ...
    if (threadIdx.x == 0) {
        __threadfence();      // ... whose (cumulative) fence publishes them before the ticket
        const unsigned int g = blockIdx.x >> 5, ngroups = (gridDim.x + 31) >> 5;
        const unsigned int gsize = min(32u, gridDim.x - g * 32);
        int last = 0;
        if (atomicAdd(&tickets[1 + g], 1u) == gsize - 1) {
            tickets[1 + g] = 0;
            __threadfence();
            if (atomicAdd(&tickets[0], 1u) == ngroups - 1) { tickets[0] = 0; last = 1; }
        }
        *s_flag = last;
    }
    __syncthreads();
    if (*s_flag) __threadfence();
    return *s_flag != 0;
}

// Sum of up to 3 partial arrays (counts <= 8 * blockDim) with all loads in flight at once.
__device__ __forceinline__ void reduce3_cg(const double* a, int na, const double* b, int nb, const double* c,
                                           int nc, double* smem, double& sa, double& sb, double& sc) {
    double va[8], vb[8], vc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = threadIdx.x + k * blockDim.x;
        va[k] = i < na ? __ldcg(&a[i]) : 0.0;
        vb[k] = i < nb ? __ldcg(&b[i]) : 0.0;
        vc[k] = i < nc ? __ldcg(&c[i]) : 0.0;
    }
    double ta = 0.0, tb = 0.0, tc = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { ta += va[k]; tb += vb[k]; tc += vc[k]; }
    sa = block_sum(ta, smem);
    sb = block_sum(tb, smem);
    sc = block_sum(tc, smem);
}

// Vector pass of the fused iteration.  The first `nbc` CTAs start with the boundary rows (the
// rows some peer needs): update them, store the new u entries straight into the peers' halo
// tails, and the last of them to finish raises this rank's flag in the peers' mailboxes and
// waits for theirs -- so the halo exchange runs under the bulk of the kernel, and the kernel
// cannot complete before this rank's halo is valid.  Then every CTA does its share of the
// regular grid-stride update, skipping the boundary rows (bmask).
template <bool UNIT>
__global__ void __launch_bounds__(PCG_THREADS)
dist_vector_push_kernel(PcgDev* __restrict__ dev, int32_t n, double* __restrict__ cur, const double* __restrict__ prev,
                        double* __restrict__ x, double* __restrict__ r, double* __restrict__ p,
                        double* __restrict__ s, const double* __restrict__ w, const double* __restrict__ dinv,
                        double* u, double* __restrict__ part_g, double* __restrict__ part_rr,
                        DistSync* sy, const unsigned long long* __restrict__ seq, int R, int me,
                        const int32_t* __restrict__ send_idx, const int32_t* __restrict__ send_off,
                        const long long* __restrict__ dest_off, const int32_t* __restrict__ need_cnt,
                        const int32_t* __restrict__ blist, int nb, int nbc, const int32_t* __restrict__ push_rng,
                        const unsigned char* __restrict__ bmask, char* const* __restrict__ peer) {
    __shared__ double sm[40];
    __shared__ int s_last;
    if (block_done(&dev->done)) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long now = gtime();
        if (sy->dbg[10]) { sy->dbg[11] += now - sy->dbg[10]; }   // end of previous S tail -> this V start
        sy->dbg[8] = now;
    }
    const double g = cur[0], dl = cur[1], rr = cur[2];
    const double gp = prev[0], ap = prev[3];
    const bool conv = rr <= dev->tol2;
    double beta = 0.0, den = dl;
    if (ap != 0.0) { beta = g / gp; den = dl - beta * g / ap; }
    const double alpha = g / den;
    const bool bad = !(den > 0.0) || !(rr == rr);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        dev->rr = rr;
        if (conv) { dev->done = 1; dev->status = NODAL_OK; }
        else if (bad) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
        else { dev->iters = dev->iters + 1; cur[3] = alpha; }
    }
    if (conv || bad) return;
    double lg = 0.0, lrr = 0.0;
    if ((int)blockIdx.x < nbc) {
        // ---------------- boundary rows first ----------------
        const unsigned long long tv0 = gtime();
        const int chunk = (nb + nbc - 1) / nbc;
        const int k0 = blockIdx.x * chunk, k1 = min(nb, k0 + chunk);
        for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
            const int i = blist[k];
            const double dvi = UNIT ? 1.0 : dinv[i];
            const double pv = fma(beta, p[i], dvi * r[i]);
            const double sv = fma(beta, s[i], w[i]);
            const double rv = fma(-alpha, sv, r[i]);
            p[i] = pv; s[i] = sv; x[i] = fma(alpha, pv, x[i]); r[i] = rv;
            if (!UNIT) { const double uv = dvi * rv; u[i] = uv; lg = fma(rv, uv, lg); }
            lrr = fma(rv, rv, lrr);
        }
        __syncthreads();
        const double* src = UNIT ? r : u;    // what the peers gather: r itself when the diagonal is 1
        // entries of the (sorted) send lists that reference my rows: ranges precomputed on the host
        for (int o = 0; o < R; ++o) {
            if (o == me) continue;
            const int b = send_off[o];
            const int first = push_rng[(blockIdx.x * R + o) * 2], last = push_rng[(blockIdx.x * R + o) * 2 + 1];
            double* dst = reinterpret_cast<double*>(peer[o] + P2P_HDR) + dest_off[o];
            for (int j = first + threadIdx.x; j < last; j += blockDim.x) dst[j - b] = src[send_idx[j]];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();   // cumulative: covers the whole CTA's local and remote stores
            const unsigned int t = atomicAdd(&sy->ticket_v[0], 1u);
            s_last = (t == (unsigned int)nbc - 1);
            if (s_last) sy->ticket_v[0] = 0;
        }
        __syncthreads();
        if (s_last) {
            __threadfence_system();
            const unsigned long long tv1 = gtime();
            const unsigned long long tag = *seq + 1;
            P2PMail* mine = reinterpret_cast<P2PMail*>(peer[me]);
            if (threadIdx.x < R && threadIdx.x != me) {
                if (send_off[threadIdx.x + 1] > send_off[threadIdx.x]) {
                    P2PMail* m = reinterpret_cast<P2PMail*>(peer[threadIdx.x]);
                    st_sys_u64(&m->hflag[me], tag);
                }
                if (need_cnt[threadIdx.x] > 0) {
                    const long long t0 = clock64();
                    while (ld_sys_u64(&mine->hflag[threadIdx.x]) < tag) {
                        if (clock64() - t0 > P2P_SPIN_LIMIT) {
                            dev->done = 1; dev->status = NODAL_CUDA_ERROR; mine->err = 1;
                            break;
                        }
                    }
                }
            }
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                const unsigned long long tv2 = gtime();
                sy->dbg[0] += tv1 - tv0; sy->dbg[1] += tv2 - tv1; sy->dbg[2] += 1;
            }
        }
    }
    {
        // ---------------- regular grid-stride share ----------------
        const int64_t n2 = n >> 1;
        const int64_t stride = (int64_t)gridDim.x * blockDim.x;
        double2* x2 = reinterpret_cast<double2*>(x);
        double2* r2 = reinterpret_cast<double2*>(r);
        double2* p2 = reinterpret_cast<double2*>(p);
        double2* s2 = reinterpret_cast<double2*>(s);
        double2* u2 = reinterpret_cast<double2*>(u);
        const double2* w2 = reinterpret_cast<const double2*>(w);
        const double2* d2 = reinterpret_cast<const double2*>(dinv);
        const uchar2* m2 = reinterpret_cast<const uchar2*>(bmask);
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
            const uchar2 mk = m2[i];
            double2 xv = x2[i], rv = r2[i], pv = p2[i], sv = s2[i];
            const double2 wv = w2[i];
            double2 dv = make_double2(1.0, 1.0);
            if (!UNIT) dv = d2[i];
            if (mk.x | mk.y) {   // a boundary row in this pair: element-wise, skipping the rows done above
                if (!mk.x) {
                    pv.x = fma(beta, pv.x, dv.x * rv.x); sv.x = fma(beta, sv.x, wv.x);
                    xv.x = fma(alpha, pv.x, xv.x); rv.x = fma(-alpha, sv.x, rv.x);
                    p[2 * i] = pv.x; s[2 * i] = sv.x; x[2 * i] = xv.x; r[2 * i] = rv.x;
                    if (!UNIT) { const double uv = dv.x * rv.x; u[2 * i] = uv; lg = fma(rv.x, uv, lg); }
                    lrr = fma(rv.x, rv.x, lrr);
                }
                if (!mk.y) {
                    pv.y = fma(beta, pv.y, dv.y * rv.y); sv.y = fma(beta, sv.y, wv.y);
                    xv.y = fma(alpha, pv.y, xv.y); rv.y = fma(-alpha, sv.y, rv.y);
                    p[2 * i + 1] = pv.y; s[2 * i + 1] = sv.y; x[2 * i + 1] = xv.y; r[2 * i + 1] = rv.y;
                    if (!UNIT) { const double uv = dv.y * rv.y; u[2 * i + 1] = uv; lg = fma(rv.y, uv, lg); }
                    lrr = fma(rv.y, rv.y, lrr);
                }
                continue;
            }
            pv.x = fma(beta, pv.x, dv.x * rv.x); pv.y = fma(beta, pv.y, dv.y * rv.y);
            sv.x = fma(beta, sv.x, wv.x);        sv.y = fma(beta, sv.y, wv.y);
            xv.x = fma(alpha, pv.x, xv.x);       xv.y = fma(alpha, pv.y, xv.y);
            rv.x = fma(-alpha, sv.x, rv.x);      rv.y = fma(-alpha, sv.y, rv.y);
            p2[i] = pv; s2[i] = sv; x2[i] = xv; r2[i] = rv;
            if (!UNIT) {
                double2 uv;
                uv.x = dv.x * rv.x; uv.y = dv.y * rv.y;
                u2[i] = uv;
                lg = fma(rv.x, uv.x, lg); lg = fma(rv.y, uv.y, lg);
            }
            lrr = fma(rv.x, rv.x, lrr); lrr = fma(rv.y, rv.y, lrr);
        }
        if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0 && !bmask[n - 1]) {
            const int64_t i = n - 1;
            const double dvi = UNIT ? 1.0 : dinv[i];
            const double pv = fma(beta, p[i], dvi * r[i]);
            const double sv = fma(beta, s[i], w[i]);
            const double rv = fma(-alpha, sv, r[i]);
            p[i] = pv; s[i] = sv; x[i] = fma(alpha, pv, x[i]); r[i] = rv;
            if (!UNIT) { const double uv = dvi * rv; u[i] = uv; lg = fma(rv, uv, lg); }
            lrr = fma(rv, rv, lrr);
        }
    }
    lrr = block_sum(lrr, sm);
    lg = UNIT ? lrr : block_sum(lg, sm);
    if (threadIdx.x == 0) { part_g[blockIdx.x] = lg; part_rr[blockIdx.x] = lrr; }
}

// SpMV of the fused iteration; the CTA that finishes last runs the all-reduce through the
// peers' mailboxes (fixed reduction order: the result does not depend on which CTA is last).
template <class A>
__global__ void __launch_bounds__(PCG_THREADS, 5)
dist_spmv_allreduce_sell_kernel(PcgDev* __restrict__ dev, int32_t n, int32_t nslices,
                                const u32* __restrict__ slice_w, A a0, const double* __restrict__ u,
                                double* __restrict__ w, double* part_d, const double* __restrict__ part_g,
                                const double* __restrict__ part_rr, int cnt_v, DistSync* sy,
                                unsigned long long* seq, int R, int me,
                                char* const* __restrict__ peer, double* __restrict__ out) {
    __shared__ double sm[40];
    __shared__ double s_slot[P2P_MAXR][3];
    __shared__ int s_flag;
    if (block_done(&dev->done)) return;
    const unsigned long long s0 = *seq;
    const unsigned long long tag = s0 + 1;
    P2PMail* mine = reinterpret_cast<P2PMail*>(peer[me]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long now = gtime();
        sy->dbg[12] += now - sy->dbg[8];    // V start -> S start
        sy->dbg[9] = now;
    }
    // (the halo part of u is complete: dist_vector_push_kernel does not finish before it is)
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double dot = 0.0;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int wd = (int)(slice_w[s + 1] - w0);
        const int64_t base = (int64_t)w0 * 32 + lane;
        const int64_t row = s * 32 + lane;
        const double acc = sell_row_dot(a, base, row, wd, u);
        if (row < n) {
            w[row] = acc;
            dot = fma(acc, __ldg(&u[row]), dot);
        }
    }
    dot = block_sum(dot, sm);
    if (threadIdx.x == 0) part_d[blockIdx.x] = dot;
    if (!last_cta_arrive(sy->ticket_s, &s_flag)) return;
    const unsigned long long ts0 = gtime();
    double g, rr, dl;
    reduce3_cg(part_g, cnt_v, part_rr, cnt_v, part_d, (int)gridDim.x, sm, g, rr, dl);
    const int par = (int)(s0 & 1ull);
    __syncthreads();
    if (threadIdx.x == 0) s_flag = 0;
    __syncthreads();
    const unsigned long long ts1 = gtime();
    unsigned long long ts2 = ts1;
    if (threadIdx.x < R) {
        P2PMail* m = reinterpret_cast<P2PMail*>(peer[threadIdx.x]);
        volatile double* slot = m->red[par][me];
        slot[0] = g; slot[1] = dl; slot[2] = rr;
        st_sys_u64(reinterpret_cast<unsigned long long*>(&m->red[par][me][3]), tag);   // release: data first
        ts2 = gtime();
        const unsigned long long* tp = reinterpret_cast<const unsigned long long*>(&mine->red[par][threadIdx.x][3]);
        const long long t0 = clock64();
        while (ld_sys_u64(tp) != tag) {
            if (clock64() - t0 > P2P_SPIN_LIMIT) { s_flag = 1; break; }
        }
        const volatile double* in = mine->red[par][threadIdx.x];
        s_slot[threadIdx.x][0] = in[0]; s_slot[threadIdx.x][1] = in[1]; s_slot[threadIdx.x][2] = in[2];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_flag) {
            dev->done = 1; dev->status = NODAL_CUDA_ERROR; mine->err = 1;
        } else {
            double sg = 0.0, sd = 0.0, sr = 0.0;
            for (int t = 0; t < R; ++t) { sg += s_slot[t][0]; sd += s_slot[t][1]; sr += s_slot[t][2]; }
            out[0] = sg; out[1] = sd; out[2] = sr;
            *seq = tag;
            if (dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        }
        const unsigned long long ts3 = gtime();
        sy->dbg[4] += ts1 - ts0; sy->dbg[5] += ts2 - ts1; sy->dbg[6] += ts3 - ts2; sy->dbg[7] += 1;
        sy->dbg[13] += ts0 - sy->dbg[9];    // S start -> S tail begin
        sy->dbg[10] = ts3;
    }
}

__global__ void __launch_bounds__(DT)
dist_mark_rows_kernel(int64_t m, const int32_t* __restrict__ rows, unsigned char* __restrict__ mask) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        mask[rows[i]] = 1;
}

static int grid_of(nodal_ctx* ctx, int64_t work) {
    int64_t b = (work + DT - 1) / DT;
    const int64_t cap = (int64_t)ctx->num_sms * 8;
    return (int)std::max<int64_t>(1, std::min(b, cap));
}

int peer_heap_ensure(nodal_ctx* ctx, nodal_dist* d, PeerHeap* hp, size_t bytes, size_t zero_bytes,
                     cudaStream_t st, bool* usable) {
    *usable = false;
    const int R = d->nranks, me = d->rank;
    if (R < 2 || R > P2P_MAXR || d->p2p_disabled || getenv("NODAL_DIST_NO_P2P")) return NODAL_OK;
    int* flag_dev = nullptr;
    CUDA_TRY(cudaMalloc(&flag_dev, 256));
    int ok = 1;
    if (hp->bytes < bytes) {
        CUDA_TRY(cudaStreamSynchronize(st));
        peer_heap_release(d, hp);
        const size_t want = align_up(bytes + bytes / 4, 2 << 20);
        cudaIpcMemHandle_t mine;
        char* handles_dev = nullptr;
        std::vector<cudaIpcMemHandle_t> all((size_t)R);
        if (cudaMalloc(&hp->shm, want) != cudaSuccess) ok = 0;
        if (ok && cudaMemset(hp->shm, 0, std::min(zero_bytes, want)) != cudaSuccess) ok = 0;
        if (ok && cudaIpcGetMemHandle(&mine, hp->shm) != cudaSuccess) ok = 0;
        if (!ok) memset(&mine, 0, sizeof(mine));
        (void)cudaGetLastError();
        CUDA_TRY(cudaMalloc(&handles_dev, sizeof(cudaIpcMemHandle_t) * (size_t)(R + 1)));
        CUDA_TRY(cudaMemcpy(handles_dev + sizeof(cudaIpcMemHandle_t) * (size_t)R, &mine, sizeof(mine), cudaMemcpyHostToDevice));
        NCCL_TRY(g_nccl.AllGather(handles_dev + sizeof(cudaIpcMemHandle_t) * (size_t)R, handles_dev,
                                  sizeof(cudaIpcMemHandle_t), ncclChar, d->comm, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemcpy(all.data(), handles_dev, sizeof(cudaIpcMemHandle_t) * (size_t)R, cudaMemcpyDeviceToHost));
        cudaFree(handles_dev);
        hp->peer.assign((size_t)R, nullptr);
        for (int o = 0; o < R && ok; ++o) {
            if (o == me) { hp->peer[o] = hp->shm; continue; }
            void* ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, all[o], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                ok = 0;
                (void)cudaGetLastError();
            }
            hp->peer[o] = static_cast<char*>(ptr);
        }
        if (ok) {
            if (cudaMalloc(&hp->peer_dev, sizeof(char*) * P2P_MAXR) != cudaSuccess ||
                cudaMemcpy(hp->peer_dev, hp->peer.data(), sizeof(char*) * (size_t)R, cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMalloc(&hp->seq, 256) != cudaSuccess || cudaMemset(hp->seq, 0, 256) != cudaSuccess)
                ok = 0;
        }
        if (ok) hp->bytes = want;
    }
    // agree on the outcome (also a barrier: nobody writes a mailbox before it has been zeroed)
    CUDA_TRY(cudaMemcpy(flag_dev, &ok, sizeof(int), cudaMemcpyHostToDevice));
    NCCL_TRY(g_nccl.AllReduce(flag_dev, flag_dev, 1, ncclInt32, ncclMin, d->comm, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    int all_ok = 0;
    CUDA_TRY(cudaMemcpy(&all_ok, flag_dev, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(flag_dev);
    if (!all_ok) {
        peer_heap_release(d, hp);
        d->p2p_disabled = true;
        return NODAL_OK;
    }
    *usable = true;
    return NODAL_OK;
}

extern "C" int nodal_dist_pcg(nodal_ctx* ctx, nodal_dist* d, int32_t n_global, const int32_t* bounds_h,
                              int64_t nnz, const int32_t* indptr, const int32_t* indices,
                              const double* data, const double* rhs_local, double* x_local,
                              double rtol, int32_t maxit, int32_t* iters_h, double* relres_h,
                              double* stats_h, void* stream) {
    NvtxRange nvtx_range("nodal_dist_pcg");
    if (!ctx || !d || !bounds_h || !iters_h || !relres_h) return NODAL_BAD_ARG;
    if (!d->comm) {
        nodal_set_error("nodal_dist_pcg needs a communicator (nodal_dist_create); use nodal_pcg on one GPU");
        return NODAL_BAD_ARG;
    }
    *iters_h = 0;
    *relres_h = 0.0;
    if (stats_h) memset(stats_h, 0, 16 * sizeof(double));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int R = d->nranks, me = d->rank;
    const int32_t rb = bounds_h[me], re = bounds_h[me + 1];
    const int32_t nloc = re - rb;
    if (nloc <= 0 || bounds_h[0] != 0 || bounds_h[R] != n_global) {
        nodal_set_error("nodal_dist_pcg: every rank must own at least one row and bounds must span [0, n)");
        return NODAL_BAD_ARG;
    }
    cudaEvent_t ev0, ev1, ev2, ev_poll[2];
    CUDA_TRY(cudaEventCreate(&ev0));
    CUDA_TRY(cudaEventCreate(&ev1));
    CUDA_TRY(cudaEventCreate(&ev2));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[0], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[1], cudaEventDisableTiming));
    nodal_sell* sell = nullptr;
    std::vector<void*> owned;   // cudaMalloc'ed buffers that outlive the arena resets
    auto dmalloc = [&](size_t bytes) -> void* {
        void* p = ctx_pool_alloc(ctx, bytes);
        if (p) owned.push_back(p);
        return p;
    };
    PcgDev host{};
    int restarts = 0;
    float ms_setup = 0.f, ms_solve = 0.f;
    int64_t halo_total = 0, send_total = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t gexec = nullptr;
    cudaStream_t cap = nullptr;
    unsigned long long launches_per_chunk = 0;
    double host_ms_capture = 0.0;
    bool used_p2p = false;
    double* sc = nullptr;
    double un_rr = 0.0, un_bb = 0.0;

    auto run = [&]() -> int {
        CUDA_TRY(cudaEventRecord(ev0, st));
        // ---------------- halo discovery (device) ----------------
        const size_t need = align_up((size_t)nnz * 4, 256) * 2 + align_up((size_t)nnz * 8, 256) * 4 +
                            radix_sort_scratch_bytes(std::max<int64_t>(nnz, 1)) +
                            2 * scan_scratch_bytes(std::max<int64_t>(nnz, 1)) + (1 << 16);
        NODAL_TRY(ctx_reserve(ctx, need));
        u32* flag = carve<u32>(ctx, (size_t)std::max<int64_t>(nnz, 1));
        u32* tot = carve<u32>(ctx, 16);
        if (!flag || !tot) return NODAL_CUDA_ERROR;
        u32* host_tot = reinterpret_cast<u32*>(ctx->pinned);
        const int gnz = grid_of(ctx, nnz);
        int64_t next = 0, nhalo = 0;
        int32_t* halo = nullptr;
        if (nnz > 0) {
            dist_flag_external_kernel<<<gnz, DT, 0, st>>>(nnz, indices, rb, re, flag);
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
            dist_compact_external_kernel<<<gnz, DT, 0, st>>>(nnz, indices, rb, re, flag, keys);
            KERNEL_CHECK();
            int bits = 1;
            while (((int64_t)n_global >> bits) != 0) ++bits;
            bool in_alt = false;
            const size_t mark = ctx->arena_used;
            NODAL_TRY(radix_sort_pairs(ctx, keys, vals, keys_alt, vals_alt, next, bits, &in_alt, st));
            ctx->arena_used = mark;
            const u64* sk = in_alt ? keys_alt : keys;
            dist_unique_flag_kernel<<<grid_of(ctx, next), DT, 0, st>>>(next, sk, uflag);
            KERNEL_CHECK();
            NODAL_TRY(scan_exclusive_u32(ctx, uflag, uflag, next, tot, st));
            ctx->arena_used = mark;
            CUDA_TRY(cudaMemcpyAsync(host_tot, tot, sizeof(u32), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            nhalo = host_tot[0];
            halo = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)nhalo));
            if (!halo) return NODAL_CUDA_ERROR;
            dist_unique_compact_kernel<<<grid_of(ctx, next), DT, 0, st>>>(next, sk, uflag, halo);
            KERNEL_CHECK();
        }
        halo_total = nhalo;
        int32_t* lcols = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)std::max<int64_t>(nnz, 1)));
        if (!lcols) return NODAL_CUDA_ERROR;
        if (nnz > 0) {
            dist_remap_kernel<<<gnz, DT, 0, st>>>(nnz, indices, rb, re, halo, (int32_t)nhalo, lcols);
            KERNEL_CHECK();
        }
        // ---------------- who needs what (host bookkeeping of <= R counts) ----------------
        std::vector<int32_t> halo_h((size_t)nhalo);
        if (nhalo) CUDA_TRY(cudaMemcpyAsync(halo_h.data(), halo, sizeof(int32_t) * (size_t)nhalo, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        std::vector<int32_t> need_from(R, 0), need_off(R + 1, 0);
        {
            int o = 0;
            for (int64_t i = 0; i < nhalo; ++i) {
                while (halo_h[i] >= bounds_h[o + 1]) ++o;
                need_from[o]++;
            }
            for (int o2 = 0; o2 < R; ++o2) need_off[o2 + 1] = need_off[o2] + need_from[o2];
        }
        const int W = R + 1;   // per rank: R counts + its u length
        int32_t* cnt_dev = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)W * (R + 1)));
        if (!cnt_dev) return NODAL_CUDA_ERROR;
        std::vector<int32_t> mine_row(W, 0);
        for (int o = 0; o < R; ++o) mine_row[o] = need_from[o];
        mine_row[R] = (int32_t)((nloc + nhalo + 2 + 255) / 256);      // u length in units of 256 doubles
        CUDA_TRY(cudaMemcpyAsync(cnt_dev + (size_t)W * R, mine_row.data(), sizeof(int32_t) * W, cudaMemcpyHostToDevice, st));
        NCCL_TRY(g_nccl.AllGather(cnt_dev + (size_t)W * R, cnt_dev, W, ncclInt32, d->comm, st));
        std::vector<int32_t> gathered((size_t)W * R);
        CUDA_TRY(cudaMemcpyAsync(gathered.data(), cnt_dev, sizeof(int32_t) * (size_t)W * R, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        std::vector<int32_t> cnt((size_t)R * R);
        int64_t max_units = 0;
        for (int s2 = 0; s2 < R; ++s2) {
            for (int o = 0; o < R; ++o) cnt[(size_t)s2 * R + o] = gathered[(size_t)s2 * W + o];
            max_units = std::max<int64_t>(max_units, gathered[(size_t)s2 * W + R]);
        }
        // cnt[s*R + o] = entries rank s needs from owner o
        std::vector<int32_t> send_cnt(R, 0), send_off(R + 1, 0);
        for (int s = 0; s < R; ++s) send_cnt[s] = cnt[(size_t)s * R + me];
        for (int s = 0; s < R; ++s) send_off[s + 1] = send_off[s] + send_cnt[s];
        send_total = send_off[R];
        int32_t* send_idx = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)std::max<int64_t>(send_total, 1)));
        double* send_buf = static_cast<double*>(dmalloc(sizeof(double) * (size_t)std::max<int64_t>(send_total, 1)));
        if (!send_idx || !send_buf) return NODAL_CUDA_ERROR;
        NCCL_TRY(g_nccl.GroupStart());
        for (int o = 0; o < R; ++o) {
            if (o == me) continue;
            if (need_from[o]) NCCL_TRY(g_nccl.Send(halo + need_off[o], need_from[o], ncclInt32, o, d->comm, st));
            if (send_cnt[o]) NCCL_TRY(g_nccl.Recv(send_idx + send_off[o], send_cnt[o], ncclInt32, o, d->comm, st));
        }
        NCCL_TRY(g_nccl.GroupEnd());
        if (send_total) {
            dist_rebase_kernel<<<grid_of(ctx, send_total), DT, 0, st>>>(send_total, send_idx, rb);
            KERNEL_CHECK();
        }
        // ---------------- peer-memory path: symmetric buffer + push metadata ----------------
        bool p2p = false;
        NODAL_TRY(peer_heap_ensure(ctx, d, &d->pcg, P2P_HDR + (size_t)max_units * 256 * sizeof(double), P2P_HDR, st, &p2p));
        int32_t* send_off_dev = nullptr;
        int32_t* need_cnt_dev = nullptr;
        long long* dest_off_dev = nullptr;
        if (p2p) {
            std::vector<long long> dest_off(R, 0);
            for (int o = 0; o < R; ++o) {
                long long off = bounds_h[o + 1] - bounds_h[o];            // peer's owned part
                for (int o2 = 0; o2 < me; ++o2) off += cnt[(size_t)o * R + o2];   // blocks of lower-ranked owners
                dest_off[o] = off;
            }
            send_off_dev = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)(R + 1)));
            need_cnt_dev = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)R));
            dest_off_dev = static_cast<long long*>(dmalloc(sizeof(long long) * (size_t)R));
            if (!send_off_dev || !need_cnt_dev || !dest_off_dev) return NODAL_CUDA_ERROR;
            CUDA_TRY(cudaMemcpyAsync(send_off_dev, send_off.data(), sizeof(int32_t) * (size_t)(R + 1), cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(need_cnt_dev, need_from.data(), sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(dest_off_dev, dest_off.data(), sizeof(long long) * (size_t)R, cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaStreamSynchronize(st));   // the host vectors above go out of scope
        }
        used_p2p = p2p;
        // boundary rows (unique, sorted) = what the communication CTA of the vector pass owns
        int32_t* blist_dev = nullptr;
        int32_t* push_rng_dev = nullptr;
        unsigned char* bmask_dev = nullptr;
        int nb_rows = 0, nbc = 1;
        if (p2p) {
            std::vector<int32_t> sidx((size_t)send_total);
            if (send_total) CUDA_TRY(cudaMemcpy(sidx.data(), send_idx, sizeof(int32_t) * (size_t)send_total, cudaMemcpyDeviceToHost));
            const std::vector<int32_t> send_h = sidx;     // per-peer blocks, each ascending
            std::sort(sidx.begin(), sidx.end());
            sidx.erase(std::unique(sidx.begin(), sidx.end()), sidx.end());
            nb_rows = (int)sidx.size();
            blist_dev = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * (size_t)std::max(nb_rows, 1)));
            bmask_dev = static_cast<unsigned char*>(dmalloc((size_t)nloc + 16));
            if (!blist_dev || !bmask_dev) return NODAL_CUDA_ERROR;
            CUDA_TRY(cudaMemsetAsync(bmask_dev, 0, (size_t)nloc + 16, st));
            // CTA c of the vector pass owns blist[c*chunk, (c+1)*chunk); which send entries are those?
            const int g2_per_sm_ = getenv("NODAL_DIST_G2") ? atoi(getenv("NODAL_DIST_G2")) : 8;
            const int g2_ = (int)std::min<int64_t>((int64_t)ctx->num_sms * g2_per_sm_,
                                                   std::max<int64_t>(1, ((nloc >> 1) + PCG_THREADS - 1) / PCG_THREADS));
            nbc = std::max(1, std::min(g2_, (nb_rows + PCG_THREADS - 1) / PCG_THREADS));
            const int chunk = (nb_rows + nbc - 1) / nbc;
            std::vector<int32_t> rng((size_t)nbc * R * 2, 0);
            for (int cta = 0; cta < nbc; ++cta) {
                const int k0 = cta * chunk, k1 = std::min(nb_rows, k0 + chunk);
                for (int o = 0; o < R; ++o) {
                    int first = send_off[o], last = send_off[o];
                    if (k0 < k1 && o != me) {
                        const auto b = send_h.begin() + send_off[o], e = send_h.begin() + send_off[o + 1];
                        first = (int)(std::lower_bound(b, e, sidx[k0]) - send_h.begin());
                        last = (int)(std::upper_bound(b, e, sidx[k1 - 1]) - send_h.begin());
                    }
                    rng[((size_t)cta * R + o) * 2] = first;
                    rng[((size_t)cta * R + o) * 2 + 1] = last;
                }
            }
            push_rng_dev = static_cast<int32_t*>(dmalloc(sizeof(int32_t) * rng.size()));
            if (!push_rng_dev) return NODAL_CUDA_ERROR;
            CUDA_TRY(cudaMemcpyAsync(push_rng_dev, rng.data(), sizeof(int32_t) * rng.size(), cudaMemcpyHostToDevice, st));
            if (nb_rows) {
                CUDA_TRY(cudaMemcpyAsync(blist_dev, sidx.data(), sizeof(int32_t) * (size_t)nb_rows, cudaMemcpyHostToDevice, st));
                dist_mark_rows_kernel<<<grid_of(ctx, nb_rows), DT, 0, st>>>(nb_rows, blist_dev, bmask_dev);
                KERNEL_CHECK();
            }
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        DistSync* sy = static_cast<DistSync*>(dmalloc(sizeof(DistSync)));
        if (!sy) return NODAL_CUDA_ERROR;
        CUDA_TRY(cudaMemsetAsync(sy, 0, sizeof(DistSync), st));
        auto exchange = [&](double* v, cudaStream_t sx) -> int {   // fills v[nloc ..) from the owners
            if (R == 1) return NODAL_OK;
            if (send_total) {
                dist_gather_kernel<<<grid_of(ctx, send_total), DT, 0, sx>>>(send_total, send_idx, v, send_buf);
                KERNEL_CHECK();
            }
            NCCL_TRY(g_nccl.GroupStart());
            for (int o = 0; o < R; ++o) {
                if (o == me) continue;
                if (send_cnt[o]) NCCL_TRY(g_nccl.Send(send_buf + send_off[o], send_cnt[o], ncclFloat64, o, d->comm, sx));
                if (need_from[o]) NCCL_TRY(g_nccl.Recv(v + nloc + need_off[o], need_from[o], ncclFloat64, o, d->comm, sx));
            }
            NCCL_TRY(g_nccl.GroupEnd());
            return NODAL_OK;
        };
        // ---------------- symmetric diagonal scaling (all ranks or none) ----------------
        sc = static_cast<double*>(dmalloc(sizeof(double) * ((size_t)nloc + nhalo + 2) + 256));
        if (!sc) return NODAL_CUDA_ERROR;
        bool unit = false;
        if (getenv("NODAL_PCG_NO_SCALE") == nullptr) {
            int* flag = reinterpret_cast<int*>(sc + (size_t)nloc + nhalo + 2);
            CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
            pcg_scale_factors_kernel<<<grid_of(ctx, nloc), PCG_THREADS, 0, st>>>(nloc, indptr, lcols, data, sc, flag);
            KERNEL_CHECK();
            if (R > 1) NCCL_TRY(g_nccl.AllReduce(flag, flag, 1, ncclInt32, ncclMax, d->comm, st));
            int* flag_h = reinterpret_cast<int*>(ctx->pinned);
            CUDA_TRY(cudaMemcpyAsync(flag_h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            unit = (*flag_h == 0);
            if (unit) NODAL_TRY(exchange(sc, st));     // scale factors of the halo columns
        }
        // ---------------- local operator in the solver-private layout ----------------
        NODAL_TRY(sell_from_csr(ctx, nloc, nnz, indptr, lcols, data, &sell, st, unit ? sc : nullptr));   // resets the arena
        Mat A;
        A.n = nloc; A.nnz = nnz; A.indptr = indptr; A.indices = lcols; A.data = data;
        const double mean = (double)nnz / nloc;
        A.tpr = mean <= 2.5 ? 2 : mean <= 6.0 ? 4 : mean <= 12.0 ? 8 : mean <= 24.0 ? 16 : 32;
        bool use_sell = (double)sell->padded <= 1.5 * (double)nnz + 1024.0;
        if (R > 1) {
            // every rank must take the same path (the scaled operator exists only as SELL): agree
            int* agree = reinterpret_cast<int*>(sc + (size_t)nloc + nhalo + 2) + 4;
            const int mine = use_sell ? 1 : 0;
            CUDA_TRY(cudaMemcpyAsync(agree, &mine, sizeof(int), cudaMemcpyHostToDevice, st));
            NCCL_TRY(g_nccl.AllReduce(agree, agree, 1, ncclInt32, ncclMin, d->comm, st));
            int* agree_h = reinterpret_cast<int*>(ctx->pinned) + 8;
            CUDA_TRY(cudaMemcpyAsync(agree_h, agree, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            use_sell = *agree_h != 0;
        }
        if (use_sell) A.sell = sell;
        else unit = false;      // too irregular for SELL-32 (padding > 1.5x): CSR kernels on the unscaled operator
        const int g2_per_sm = getenv("NODAL_DIST_G2") ? atoi(getenv("NODAL_DIST_G2")) : 8;
        const int g2 = (int)std::min<int64_t>((int64_t)ctx->num_sms * g2_per_sm,
                                              std::max<int64_t>(1, ((nloc >> 1) + PCG_THREADS - 1) / PCG_THREADS));
        if (A.sell) {
            const int64_t want = ((int64_t)sell->nslices * 32 + PCG_THREADS - 1) / PCG_THREADS;
            const int per_sm = getenv("NODAL_SPMV_CTAS_PER_SM") ? atoi(getenv("NODAL_SPMV_CTAS_PER_SM")) : 5;
            A.g1 = (int)std::min<int64_t>((int64_t)ctx->num_sms * per_sm, want);
        } else {
            const int64_t want = ((int64_t)nloc * A.tpr + PCG_THREADS - 1) / PCG_THREADS;
            A.g1 = (int)std::min<int64_t>((int64_t)ctx->num_sms * 8, want);
        }
        const bool fused = p2p && A.sell && getenv("NODAL_DIST_NO_FUSE") == nullptr;
        const int gmax = std::max(A.g1, g2) + 1;
        const size_t vloc = align_up(sizeof(double) * (size_t)nloc, 256);
        const size_t vext = align_up(sizeof(double) * (size_t)(nloc + nhalo + 2), 256);
        NODAL_TRY(ctx_reserve(ctx, 7 * vloc + 2 * vext + 8 * align_up(sizeof(double) * gmax, 256) + 8192));
        // the vector the SpMV gathers from lives in the layout [owned | halo] (in the peer-mapped
        // buffer on the p2p path): u = D^-1 r in general, r itself when the diagonal is 1
        double* ext = p2p ? reinterpret_cast<double*>(d->pcg.shm + P2P_HDR)
                          : carve<double>(ctx, (size_t)nloc + nhalo + 2);
        double* r = unit ? ext : carve<double>(ctx, nloc);
        double* u = ext;
        double* q = carve<double>(ctx, nloc);                           // A x (residual checks)
        double* p = carve<double>(ctx, nloc);
        double* s = carve<double>(ctx, nloc);                           // s = A p (recurrence)
        double* w = carve<double>(ctx, nloc);                           // w = A u
        double* bh = unit ? carve<double>(ctx, nloc) : nullptr;         // S b
        if (unit && !bh) return NODAL_CUDA_ERROR;
        double* xe = carve<double>(ctx, (size_t)nloc + nhalo + 2);      // x in the same layout
        double* part_g = carve<double>(ctx, gmax);
        double* part_d = carve<double>(ctx, gmax);
        double* part_rr = carve<double>(ctx, gmax);
        double* part_bb = carve<double>(ctx, gmax);
        double* SC = carve<double>(ctx, 16);    // SC[par*4 + {gamma, delta, rr, alpha}]
        PcgDev* dev = carve<PcgDev>(ctx, 1);
        double* dinv_own = A.sell ? nullptr : carve<double>(ctx, nloc);
        if (!r || !q || !p || !s || !w || !u || !xe || !part_bb || !SC || !dev) return NODAL_CUDA_ERROR;
        const double* dinv = A.sell ? sell->dinv : dinv_own;
        if (dinv_own) {
            csr_dinv_kernel<<<g2, PCG_THREADS, 0, st>>>(nloc, indptr, lcols, data, dinv_own);
            KERNEL_CHECK();
        }
        CUDA_TRY(cudaMemsetAsync(dev, 0, sizeof(PcgDev), st));
        CUDA_TRY(cudaMemsetAsync(SC, 0, sizeof(double) * 16, st));
        const double* b_eff = rhs_local;
        if (unit) {
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(nloc, rhs_local, sc, bh, 0);       // b_hat = S b
            KERNEL_CHECK();
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(nloc, x_local, sc, x_local, 1);    // x_hat = S^-1 x0
            KERNEL_CHECK();
            b_eff = bh;
        }

        auto spmv_plain = [&](const double* in, double* out) -> int {
            if (A.sell) return nodal_sell_spmv(ctx, A.sell, in, out, st);
            return csr_spmv_launch(ctx, nloc, nnz, indptr, lcols, data, in, out, st);
        };
        // (re)start from the current x: r = b - A x, u = D^-1 r, w = A u, p = s = 0
        auto start = [&](int first) -> int {
            cgcg_reset_kernel<<<1, 32, 0, st>>>(dev);
            KERNEL_CHECK();
            CUDA_TRY(cudaMemcpyAsync(xe, x_local, sizeof(double) * (size_t)nloc, cudaMemcpyDeviceToDevice, st));
            NODAL_TRY(exchange(xe, st));
            NODAL_TRY(spmv_plain(xe, q));
            if (unit)
                cgcg_start_kernel<true><<<g2, PCG_THREADS, 0, st>>>(nloc, b_eff, q, dinv, r, u, p, s, part_g, part_rr, part_bb);
            else
                cgcg_start_kernel<false><<<g2, PCG_THREADS, 0, st>>>(nloc, b_eff, q, dinv, r, u, p, s, part_g, part_rr, part_bb);
            KERNEL_CHECK();
            NODAL_TRY(exchange(ext, st));
            NODAL_TRY(launch_k1(A, dev, ext, w, part_d, st));
            cgcg_reduce_kernel<<<1, PCG_THREADS, 0, st>>>(dev, part_g, part_rr, part_bb, g2, part_d, A.g1, SC, 1);
            KERNEL_CHECK();
            if (R > 1) NCCL_TRY(g_nccl.AllReduce(SC, SC, 4, ncclFloat64, ncclSum, d->comm, st));
            cgcg_scalars_kernel<<<1, 32, 0, st>>>(dev, SC, rtol, maxit, first);
            KERNEL_CHECK();
            return NODAL_OK;
        };
        auto iteration = [&](int par, cudaStream_t sx) -> int {
            double* cur = SC + par * 4;
            double* nxt = SC + (par ^ 1) * 4;
            if (fused) {
                // two kernels, no NCCL: push + halo wait inside the vector pass, all-reduce inside the SpMV
                if (unit)
                    dist_vector_push_kernel<true><<<g2, PCG_THREADS, 0, sx>>>(
                        dev, nloc, cur, nxt, x_local, r, p, s, w, dinv, u, part_g, part_rr, sy, d->pcg.seq, R, me,
                        send_idx, send_off_dev, dest_off_dev, need_cnt_dev, blist_dev, nb_rows, nbc, push_rng_dev,
                        bmask_dev, d->pcg.peer_dev);
                else
                    dist_vector_push_kernel<false><<<g2, PCG_THREADS, 0, sx>>>(
                        dev, nloc, cur, nxt, x_local, r, p, s, w, dinv, u, part_g, part_rr, sy, d->pcg.seq, R, me,
                        send_idx, send_off_dev, dest_off_dev, need_cnt_dev, blist_dev, nb_rows, nbc, push_rng_dev,
                        bmask_dev, d->pcg.peer_dev);
                KERNEL_CHECK();
                sell_launch(sell, [&](auto a) {
                    dist_spmv_allreduce_sell_kernel<<<A.g1, PCG_THREADS, 0, sx>>>(
                        dev, nloc, sell->nslices, sell->slice_w, a, ext, w, part_d, part_g, part_rr, g2, sy,
                        d->pcg.seq, R, me, d->pcg.peer_dev, nxt);
                });
                KERNEL_CHECK();
                return NODAL_OK;
            }
            if (unit)
                cgcg_vector_kernel<true><<<g2, PCG_THREADS, 0, sx>>>(dev, nloc, cur, nxt, x_local, r, p, s, w, dinv, u,
                                                                    part_g, part_rr);
            else
                cgcg_vector_kernel<false><<<g2, PCG_THREADS, 0, sx>>>(dev, nloc, cur, nxt, x_local, r, p, s, w, dinv, u,
                                                                     part_g, part_rr);
            KERNEL_CHECK();
            if (p2p) {
                p2p_push_kernel<<<1, 1024, 0, sx>>>(dev, d->pcg.seq, R, me, send_idx, send_off_dev, dest_off_dev,
                                                    d->pcg.peer_dev, ext);
                KERNEL_CHECK();
                p2p_wait_halo_kernel<<<1, 32, 0, sx>>>(dev, d->pcg.seq, R, me, need_cnt_dev,
                                                       reinterpret_cast<P2PMail*>(d->pcg.shm));
                KERNEL_CHECK();
            } else {
                NODAL_TRY(exchange(ext, sx));
            }
            NODAL_TRY(launch_k1(A, dev, ext, w, part_d, sx));
            if (p2p) {
                p2p_reduce_kernel<<<1, PCG_THREADS, 0, sx>>>(dev, d->pcg.seq, R, me, part_g, part_rr, g2, part_d, A.g1,
                                                            d->pcg.peer_dev, nxt);
                KERNEL_CHECK();
            } else {
                cgcg_reduce_kernel<<<1, PCG_THREADS, 0, sx>>>(dev, part_g, part_rr, nullptr, g2, part_d, A.g1, nxt, 0);
                KERNEL_CHECK();
                if (R > 1) NCCL_TRY(g_nccl.AllReduce(nxt, nxt, 3, ncclFloat64, ncclSum, d->comm, sx));
            }
            return NODAL_OK;
        };

        NODAL_TRY(start(1));
        const int CH = 32;
        const bool use_graph = getenv("NODAL_DIST_NO_GRAPH") == nullptr;
        if (use_graph) {
            const auto c0 = std::chrono::steady_clock::now();
            const unsigned long long before = g_nodal_launches;
            CUDA_TRY(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
            if (A.sell) NODAL_TRY(sell_set_l2_window(ctx, A.sell, cap));
            CUDA_TRY(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
            int crc = NODAL_OK;
            for (int i = 0; i < CH && crc == NODAL_OK; ++i) crc = iteration(i & 1, cap);
            cudaError_t ce = cudaStreamEndCapture(cap, &graph);
            if (crc != NODAL_OK) return crc;
            CUDA_TRY(ce);
            CUDA_TRY(cudaGraphInstantiate(&gexec, graph, 0));
            launches_per_chunk = g_nodal_launches - before;
            g_nodal_launches = before;
            host_ms_capture = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - c0).count();
        }
        CUDA_TRY(cudaEventRecord(ev1, st));
        PcgDev* poll = reinterpret_cast<PcgDev*>(ctx->pinned);
        double last_true_rr = -1.0;
        for (;;) {
            const int64_t max_chunks = (int64_t)maxit / CH + 3;
            int64_t k = 0;
            for (;; ++k) {
                if (use_graph) {
                    CUDA_TRY(cudaGraphLaunch(gexec, st));
                    g_nodal_launches += launches_per_chunk;
                } else {
                    for (int i = 0; i < CH; ++i) NODAL_TRY(iteration(i & 1, st));
                }
                CUDA_TRY(cudaMemcpyAsync(&poll[k & 1], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaEventRecord(ev_poll[k & 1], st));
                if (k >= 1) {
                    CUDA_TRY(cudaEventSynchronize(ev_poll[(k - 1) & 1]));
                    if (poll[(k - 1) & 1].done) break;
                }
                if (k > max_chunks) break;
            }
            CUDA_TRY(cudaStreamSynchronize(st));
            host = poll[k & 1];
            if (!host.done) host.status = NODAL_NOT_CONVERGED;
            if (host.status == NODAL_BREAKDOWN) break;
            const int recurrence_status = host.status;
            const int iters_so_far = host.iters;
            NODAL_TRY(start(0));     // true residual of the current x (and a restart, if needed)
            CUDA_TRY(cudaMemcpyAsync(&poll[0], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            host = poll[0];
            host.iters = iters_so_far;
            if (unit) {
                // the contract is on the UNSCALED residual: ||b - A x|| <= rtol ||b||
                pcg_unscaled_norm_kernel<<<g2, PCG_THREADS, 0, st>>>(nloc, r, sc, rhs_local, part_rr, part_bb);
                KERNEL_CHECK();
                dist_reduce_kernel<<<1, PCG_THREADS, 0, st>>>(part_rr, part_bb, nullptr, g2, SC + 12);
                KERNEL_CHECK();
                if (R > 1) NCCL_TRY(g_nccl.AllReduce(SC + 12, SC + 12, 2, ncclFloat64, ncclSum, d->comm, st));
                double* un = reinterpret_cast<double*>(ctx->pinned) + 64;
                CUDA_TRY(cudaMemcpyAsync(un, SC + 12, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                un_rr = un[0]; un_bb = un[1];
                const double target = rtol * rtol * un_bb;
                if (host.rr <= host.tol2 && un_rr > target && recurrence_status == NODAL_OK &&
                    host.iters < host.maxit && restarts < 8) {
                    const double tol2 = host.tol2 * std::min(0.25, 0.25 * target / un_rr);
                    const int zero = 0;
                    CUDA_TRY(cudaMemcpyAsync(&dev->tol2, &tol2, sizeof(double), cudaMemcpyHostToDevice, st));
                    CUDA_TRY(cudaMemcpyAsync(&dev->done, &zero, sizeof(int), cudaMemcpyHostToDevice, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                    ++restarts;
                    continue;
                }
                if (un_rr <= target) { host.status = NODAL_OK; break; }
                if (host.rr <= host.tol2) { host.status = NODAL_NOT_CONVERGED; break; }
            }
            if (host.rr <= host.tol2) { host.status = NODAL_OK; break; }
            if (recurrence_status == NODAL_NOT_CONVERGED || host.iters >= host.maxit) {
                host.status = NODAL_NOT_CONVERGED;
                break;
            }
            if (restarts >= 8 || (last_true_rr >= 0.0 && host.rr > 0.25 * last_true_rr)) {
                host.status = NODAL_NOT_CONVERGED;
                break;
            }
            last_true_rr = host.rr;
            ++restarts;
        }
        if (unit) {
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(nloc, x_local, sc, x_local, 0);     // x = S x_hat
            KERNEL_CHECK();
        }
        if (getenv("NODAL_DIST_DEBUG")) {
            unsigned long long dbg[16];
            CUDA_TRY(cudaMemcpy(dbg, sy->dbg, sizeof(dbg), cudaMemcpyDeviceToHost));
            fprintf(stderr, "[nodal dist rank %d] V tail: push %.2f us, flag+wait %.2f us (n=%llu); S tail: reduce %.2f us, "
                    "publish %.2f us, wait+sum %.2f us (n=%llu)\n", me,
                    dbg[2] ? dbg[0] / 1e3 / dbg[2] : 0.0, dbg[2] ? dbg[1] / 1e3 / dbg[2] : 0.0, dbg[2],
                    dbg[7] ? dbg[4] / 1e3 / dbg[7] : 0.0, dbg[7] ? dbg[5] / 1e3 / dbg[7] : 0.0,
                    dbg[7] ? dbg[6] / 1e3 / dbg[7] : 0.0, dbg[7]);
            if (dbg[7])
                fprintf(stderr, "[nodal dist rank %d] per iteration: V start->S start %.2f us, S start->S tail %.2f us, "
                        "S tail end->next V start %.2f us\n", me, dbg[12] / 1e3 / dbg[7], dbg[13] / 1e3 / dbg[7],
                        dbg[11] / 1e3 / dbg[7]);
        }
        CUDA_TRY(cudaEventRecord(ev2, st));
        CUDA_TRY(cudaEventSynchronize(ev2));
        CUDA_TRY(cudaEventElapsedTime(&ms_setup, ev0, ev1));
        CUDA_TRY(cudaEventElapsedTime(&ms_solve, ev1, ev2));
        *iters_h = host.iters;
        *relres_h = host.bb > 0.0 ? sqrt(host.rr / host.bb) : 0.0;
        if (unit && un_bb > 0.0) *relres_h = sqrt(un_rr / un_bb);
        if (stats_h) {
            stats_h[0] = host.iters;
            stats_h[1] = *relres_h;
            stats_h[2] = restarts;
            stats_h[3] = ms_solve;
            stats_h[4] = ms_setup;
            stats_h[5] = A.sell ? 1.0 : 0.0;
            stats_h[6] = A.sell ? (double)sell->padded : (double)nnz;
            stats_h[7] = A.g1;
            stats_h[12] = (double)halo_total;
            stats_h[13] = (double)send_total;
            stats_h[9] = used_p2p ? (fused ? 2.0 : 1.0) : 0.0;
            stats_h[8] = unit ? 1.0 : 0.0;
        }
        return host.status;
    };
    const auto h0 = std::chrono::steady_clock::now();
    const int rc = run();
    cudaStreamSynchronize(st);
    const auto h1 = std::chrono::steady_clock::now();
    if (gexec) cudaGraphExecDestroy(gexec);
    if (graph) cudaGraphDestroy(graph);
    if (cap) { sell_clear_l2_window(cap); cudaStreamDestroy(cap); }
    const auto h2 = std::chrono::steady_clock::now();
    if (sell) sell_free(sell);
    for (void* p : owned) ctx_pool_free(ctx, p);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1); cudaEventDestroy(ev2);
    cudaEventDestroy(ev_poll[0]); cudaEventDestroy(ev_poll[1]);
    const auto h3 = std::chrono::steady_clock::now();
    if (stats_h) {
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        stats_h[14] = ms(h0, h1);       // host wall of setup + solve
        stats_h[15] = ms(h1, h2);       // graph teardown
        stats_h[11] = ms(h2, h3);       // buffer teardown
        stats_h[10] = host_ms_capture;  // graph capture + instantiate
    }
    return rc;
}
