// Kernels of the Jacobi-PCG iteration, shared by the single-GPU driver (pcg.cu) and the
// row-partitioned multi-GPU driver (dist.cu).  See pcg.cu for the algorithm notes.
#pragma once
#include "sparse.cuh"

constexpr int PCG_THREADS = 256;
constexpr int PCG_CHUNK = 64;  // iterations per graph launch (even)

struct PcgDev {
    double bb, tol2, rr;
    int iters, done, status, maxit;
};

// Block-uniform read of the sticky `done` word (it may be written by block 0 of the
// kernel that is reading it, so every thread must see the same value).
__device__ __forceinline__ bool block_done(const int* done) {
    __shared__ int s_done;
    if (threadIdx.x == 0) s_done = *reinterpret_cast<const volatile int*>(done);
    __syncthreads();
    return s_done != 0;
}

// ---------------------------------------------------------------- K1
template <int MINB, class A>
static __global__ void __launch_bounds__(PCG_THREADS, MINB)
pcg_spmv_dot_sell_kernel(const PcgDev* __restrict__ dev, int32_t n, int32_t nslices,
                         const u32* __restrict__ slice_w, A a0, const double* __restrict__ p,
                         double* __restrict__ q, double* __restrict__ part_pq) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double dot = 0.0;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int w = (int)(slice_w[s + 1] - w0);
        const int64_t base = (int64_t)w0 * 32 + lane;
        const int64_t r = s * 32 + lane;
        const double acc = sell_row_dot(a, base, r, w, p);
        if (r < n) {
            q[r] = acc;
            dot = fma(acc, __ldg(&p[r]), dot);
        }
    }
    dot = block_sum(dot, sm);
    if (threadIdx.x == 0) part_pq[blockIdx.x] = dot;
}

template <int TPR>
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_spmv_dot_csr_kernel(const PcgDev* __restrict__ dev, int32_t n,
                        const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                        const double* __restrict__ data, const double* __restrict__ p,
                        double* __restrict__ q, double* __restrict__ part_pq) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    constexpr int RPW = 32 / TPR;
    const int lane = threadIdx.x & 31, sub = lane & (TPR - 1);
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double dot = 0.0;
    for (int64_t r0 = warp * RPW; r0 < n; r0 += nwarps * RPW) {
        const int64_t row = r0 + lane / TPR;
        double acc = 0.0;
        if (row < n) {
            const int32_t e = indptr[row + 1];
            for (int32_t j = indptr[row] + sub; j < e; j += TPR)
                acc = fma(data[j], __ldg(&p[indices[j]]), acc);
        }
#pragma unroll
        for (int o = TPR >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (sub == 0 && row < n) {
            q[row] = acc;
            dot = fma(acc, __ldg(&p[row]), dot);
        }
    }
    dot = block_sum(dot, sm);
    if (threadIdx.x == 0) part_pq[blockIdx.x] = dot;
}

// ---------------------------------------------------------------- K2
// UNIT: the operator has a unit diagonal (symmetrically pre-scaled system, see pcg.cu): the
// preconditioner is the identity, dinv is never read and r.z == r.r.
template <bool UNIT>
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_update_kernel(PcgDev* __restrict__ dev, int32_t n, const double* __restrict__ part_pq, int g1,
                  const double* __restrict__ part_rz_prev, int g2, double* __restrict__ x,
                  const double* __restrict__ p, double* __restrict__ r,
                  const double* __restrict__ q, const double* __restrict__ dinv,
                  double* __restrict__ part_rz, double* __restrict__ part_rr) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    double pq, rz, unused;
    if (g1 <= 8 * PCG_THREADS && g2 <= 8 * PCG_THREADS) {
        reduce_partials3(part_pq, g1, part_rz_prev, g2, nullptr, 0, sm, pq, rz, unused);
    } else {
        pq = reduce_partials(part_pq, g1, sm);
        rz = reduce_partials(part_rz_prev, g2, sm);
    }
    if (!(pq > 0.0)) {  // not SPD (or NaN): stop, x keeps the last good iterate
        if (blockIdx.x == 0 && threadIdx.x == 0) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
        return;
    }
    const double alpha = rz / pq;
    double lrz = 0.0, lrr = 0.0;
    const int64_t n2 = n >> 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    double2* x2 = reinterpret_cast<double2*>(x);
    double2* r2 = reinterpret_cast<double2*>(r);
    const double2* p2 = reinterpret_cast<const double2*>(p);
    const double2* q2 = reinterpret_cast<const double2*>(q);
    const double2* d2 = reinterpret_cast<const double2*>(dinv);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
        double2 xv = x2[i], rv = r2[i];
        const double2 pv = p2[i], qv = q2[i];
        xv.x = fma(alpha, pv.x, xv.x); xv.y = fma(alpha, pv.y, xv.y);
        rv.x = fma(-alpha, qv.x, rv.x); rv.y = fma(-alpha, qv.y, rv.y);
        x2[i] = xv; r2[i] = rv;
        if (!UNIT) {
            const double2 dv = d2[i];
            lrz = fma(rv.x * dv.x, rv.x, lrz); lrz = fma(rv.y * dv.y, rv.y, lrz);
        }
        lrr = fma(rv.x, rv.x, lrr); lrr = fma(rv.y, rv.y, lrr);
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t i = n - 1;
        const double xv = fma(alpha, p[i], x[i]);
        const double rv = fma(-alpha, q[i], r[i]);
        x[i] = xv; r[i] = rv;
        if (!UNIT) lrz = fma(rv * dinv[i], rv, lrz);
        lrr = fma(rv, rv, lrr);
    }
    lrr = block_sum(lrr, sm);
    lrz = UNIT ? lrr : block_sum(lrz, sm);
    if (threadIdx.x == 0) { part_rz[blockIdx.x] = lrz; part_rr[blockIdx.x] = lrr; }
}

// ---------------------------------------------------------------- K3
template <bool UNIT>
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_direction_kernel(PcgDev* __restrict__ dev, int32_t n, const double* __restrict__ part_rz_prev,
                     const double* __restrict__ part_rz, const double* __restrict__ part_rr, int g2,
                     double* __restrict__ p, const double* __restrict__ r,
                     const double* __restrict__ dinv) {
    __shared__ double sm[40];
    if (block_done(&dev->done)) return;
    double rz_old, rz_new, rr;
    if (g2 <= 8 * PCG_THREADS) {
        reduce_partials3(part_rz_prev, g2, part_rz, g2, part_rr, g2, sm, rz_old, rz_new, rr);
    } else {
        rz_old = reduce_partials(part_rz_prev, g2, sm);
        rz_new = reduce_partials(part_rz, g2, sm);
        rr = reduce_partials(part_rr, g2, sm);
    }
    const bool conv = rr <= dev->tol2;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const int it = dev->iters + 1;
        dev->iters = it;
        dev->rr = rr;
        if (conv) { dev->done = 1; dev->status = NODAL_OK; }
        else if (it >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        else if (!(rr == rr)) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
    }
    if (conv) return;
    const double beta = rz_new / rz_old;
    const int64_t n2 = n >> 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    double2* p2 = reinterpret_cast<double2*>(p);
    const double2* r2 = reinterpret_cast<const double2*>(r);
    const double2* d2 = reinterpret_cast<const double2*>(dinv);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
        double2 pv = p2[i];
        double2 zv = r2[i];
        if (!UNIT) { const double2 dv = d2[i]; zv.x *= dv.x; zv.y *= dv.y; }
        pv.x = fma(beta, pv.x, zv.x);
        pv.y = fma(beta, pv.y, zv.y);
        p2[i] = pv;
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t i = n - 1;
        p[i] = fma(beta, p[i], UNIT ? r[i] : r[i] * dinv[i]);
    }
}

// ---------------------------------------------------------------- start / restart
// r = b - q (q = A x) ; p = D^-1 r ; partials of r.D^-1 r, r.r and b.b
template <bool UNIT>
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_start_kernel(int32_t n, const double* __restrict__ b, const double* __restrict__ q,
                 const double* __restrict__ dinv, double* __restrict__ r, double* __restrict__ p,
                 double* __restrict__ part_rz, double* __restrict__ part_rr,
                 double* __restrict__ part_bb) {
    __shared__ double sm[40];
    double lrz = 0.0, lrr = 0.0, lbb = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double bv = b[i];
        const double rv = bv - q[i];
        const double zv = UNIT ? rv : rv * dinv[i];
        r[i] = rv;
        p[i] = zv;
        lrz = fma(rv, zv, lrz);
        lrr = fma(rv, rv, lrr);
        lbb = fma(bv, bv, lbb);
    }
    lrz = block_sum(lrz, sm);
    lrr = block_sum(lrr, sm);
    lbb = block_sum(lbb, sm);
    if (threadIdx.x == 0) {
        part_rz[blockIdx.x] = lrz;
        part_rr[blockIdx.x] = lrr;
        part_bb[blockIdx.x] = lbb;
    }
}

static __global__ void __launch_bounds__(PCG_THREADS)
pcg_scalars_kernel(PcgDev* dev, const double* part_rr, const double* part_bb, int g2, double rtol,
                   int maxit, int first) {
    __shared__ double sm[40];
    const double rr = reduce_partials(part_rr, g2, sm);
    const double bb = reduce_partials(part_bb, g2, sm);
    if (threadIdx.x == 0) {
        if (first) {
            dev->bb = bb;
            dev->tol2 = rtol * rtol * bb;
            dev->iters = 0;
            dev->maxit = maxit;
        }
        dev->rr = rr;
        dev->status = NODAL_OK;
        dev->done = 0;
        if (rr <= dev->tol2) dev->done = 1;
        else if (dev->iters >= dev->maxit) { dev->done = 1; dev->status = NODAL_NOT_CONVERGED; }
        else if (!(rr == rr)) { dev->done = 1; dev->status = NODAL_BREAKDOWN; }
    }
}

static __global__ void __launch_bounds__(PCG_THREADS)
csr_dinv_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                const double* __restrict__ data, double* __restrict__ dinv) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n;
         r += (int64_t)gridDim.x * blockDim.x) {
        double dg = 0.0;
        for (int32_t j = indptr[r]; j < indptr[r + 1]; ++j)
            if (indices[j] == r) dg += data[j];
        dinv[r] = dg != 0.0 ? 1.0 / dg : 1.0;
    }
}


// ---------------------------------------------------------------- symmetric diagonal scaling
// sc = 1 / sqrt(diag(A)).  Jacobi-PCG on A x = b is, iterate for iterate, plain CG on
// (S A S)(S^-1 x) = S b with S = diag(sc); the scaled operator has a unit diagonal, so the
// iteration never touches a preconditioner vector (16 n fewer bytes per iteration).
// *flag is raised when a diagonal entry is not positive (then the unscaled kernels are used).
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_scale_factors_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                         const double* __restrict__ data, double* __restrict__ sc, int* __restrict__ flag) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n;
         r += (int64_t)gridDim.x * blockDim.x) {
        double dg = 0.0;
        for (int32_t j = indptr[r]; j < indptr[r + 1]; ++j)
            if (indices[j] == r) dg += data[j];
        if (dg > 0.0) sc[r] = 1.0 / sqrt(dg);
        else { sc[r] = 1.0; *flag = 1; }
    }
}

// out = in * sc (mode 0) or in / sc (mode 1); in and out may alias
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_scale_vec_kernel(int32_t n, const double* in, const double* __restrict__ sc, double* out, int mode) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        out[i] = mode ? in[i] / sc[i] : in[i] * sc[i];
}

// partial sums of the UNSCALED residual norm (r_hat / sc)^2 and of b^2
static __global__ void __launch_bounds__(PCG_THREADS)
pcg_unscaled_norm_kernel(int32_t n, const double* __restrict__ rhat, const double* __restrict__ sc,
                         const double* __restrict__ b, double* __restrict__ part_rr,
                         double* __restrict__ part_bb) {
    __shared__ double sm[40];
    double lrr = 0.0, lbb = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double rv = rhat[i] / sc[i];
        lrr = fma(rv, rv, lrr);
        lbb = fma(b[i], b[i], lbb);
    }
    lrr = block_sum(lrr, sm);
    lbb = block_sum(lbb, sm);
    if (threadIdx.x == 0) { part_rr[blockIdx.x] = lrr; part_bb[blockIdx.x] = lbb; }
}

// ---------------------------------------------------------------- operator handle
struct Mat {
    // exactly one of sell / csr is used by K1
    const nodal_sell* sell = nullptr;
    int32_t n = 0;
    int64_t nnz = 0;
    const int32_t* indptr = nullptr;
    const int32_t* indices = nullptr;
    const double* data = nullptr;
    int tpr = 4;
    int g1 = 1;
    int minb = 5;      // resident CTAs per SM the SELL kernel is compiled for
};

static inline int launch_k1(const Mat& A, const PcgDev* dev, const double* p, double* q, double* part_pq,
              cudaStream_t st) {
    if (A.sell) {
#define GOS(M)                                                                                 \
    pcg_spmv_dot_sell_kernel<M><<<A.g1, PCG_THREADS, 0, st>>>(dev, A.n, A.sell->nslices,       \
                                                              A.sell->slice_w, a, p, q, part_pq)
        sell_launch(A.sell, [&](auto a) {
            switch (A.minb) {
                case 5: GOS(5); break;
                case 6: GOS(6); break;
                default: GOS(4); break;
            }
        });
#undef GOS
    } else {
#define GO(T)                                                                                  \
    pcg_spmv_dot_csr_kernel<T><<<A.g1, PCG_THREADS, 0, st>>>(dev, A.n, A.indptr, A.indices,    \
                                                             A.data, p, q, part_pq)
        switch (A.tpr) {
            case 2: GO(2); break;
            case 4: GO(4); break;
            case 8: GO(8); break;
            case 16: GO(16); break;
            default: GO(32); break;
        }
#undef GO
    }
    KERNEL_CHECK();
    return NODAL_OK;
}
