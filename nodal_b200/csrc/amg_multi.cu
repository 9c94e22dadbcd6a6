// AMG-preconditioned CG for several right-hand sides at once (SURVEY.md section 8(f) rank 4: many-port
// equivalent resistance, nodal/equiv.py:31-61 generalised): K <= 8 independent PCG recurrences
// advanced in lockstep against ONE hierarchy, so every operator of every level is read once per
// sweep for all K vectors (SpMM-shaped kernels: `12 nnz + K (8..32) n` bytes instead of K times
// `12 nnz + (8..32) n`).  Each system keeps its own alpha / beta / stopping test; a system that has
// converged is frozen (its updates are masked), the batch stops when all have.  Per system the
// arithmetic is the single-vector path's (same kernels' row order, same cycle), so results agree
// with nodal_amg_pcg to rounding.
// Vectors of a batch are stored one after the other: vector k of a level with n rows at v + k * n.
#include <algorithm>
#include <cmath>

#include "amg_host.cuh"

namespace {

constexpr int MK = 8;      // right-hand sides per batch

// dot products of one SELL row (lane, row r) with K vectors: columns / values loaded once
template <int W, class A>
__device__ __forceinline__ void sell_dot_fixed_multi(const A& a, int64_t base, int64_t r, const double* __restrict__ x,
                                                     int64_t stride, int K, double* acc) {
    int32_t c[W];
    double v[W];
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const typename A::Entry e = a.load(base + (int64_t)i * 32);
        c[i] = a.col(e, r);
        v[i] = a.val(e);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {          // compile-time indices keep acc[] in registers
        if (k < K) {
            const double* xk = x + (int64_t)k * stride;
            double a = acc[k];
#pragma unroll
            for (int i = 0; i < W; ++i) a = fma(v[i], __ldg(&xk[c[i]]), a);
            acc[k] = a;
        }
    }
}

template <class A>
__device__ __forceinline__ void sell_row_dot_multi(const A& a, int64_t base, int64_t r, int w,
                                                   const double* __restrict__ x, int64_t stride, int K, double* acc) {
    int k = 0;
    for (; k + 4 <= w; k += 4) sell_dot_fixed_multi<4>(a, base + (int64_t)k * 32, r, x, stride, K, acc);
    const int64_t b = base + (int64_t)k * 32;
    switch (w - k) {   // warp-uniform
        case 3: sell_dot_fixed_multi<3>(a, b, r, x, stride, K, acc); break;
        case 2: sell_dot_fixed_multi<2>(a, b, r, x, stride, K, acc); break;
        case 1: sell_dot_fixed_multi<1>(a, b, r, x, stride, K, acc); break;
        default: break;
    }
}

// MODE 0: y = A x and per-block partials of x.y   MODE 1: y = b - A x   MODE 2: y = x + omega D^-1 (b - A x)
template <int MODE, class A>
__global__ void __launch_bounds__(AT, 3)
amgm_sell_kernel(int32_t n, int32_t nslices, const u32* __restrict__ slice_w, A a0, const double* __restrict__ dinv, const double* __restrict__ b,
                 const double* __restrict__ x, double omega, double* __restrict__ y, double* __restrict__ part, int K,
                 int nparts) {
    __shared__ double red[33];
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double dot[MK];
#pragma unroll
    for (int k = 0; k < MK; ++k) dot[k] = 0.0;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int w = (int)(slice_w[s + 1] - w0);
        double acc[MK];
#pragma unroll
        for (int k = 0; k < MK; ++k) acc[k] = 0.0;
        const int64_t r = s * 32 + lane;
        sell_row_dot_multi(a, (int64_t)w0 * 32 + lane, r, w, x, n, K, acc);
        if (r < n) {
            const double di = MODE == 2 ? dinv[r] : 0.0;
#pragma unroll
            for (int k = 0; k < MK; ++k) {
                if (k >= K) break;
                const int64_t o = (int64_t)k * n + r;
                if (MODE == 0) { y[o] = acc[k]; dot[k] = fma(x[o], acc[k], dot[k]); }
                if (MODE == 1) y[o] = b[o] - acc[k];
                if (MODE == 2) y[o] = x[o] + omega * di * (b[o] - acc[k]);
            }
        }
    }
    if (MODE == 0) {
#pragma unroll
        for (int k = 0; k < MK; ++k) {
            if (k < K) {                       // K is uniform over the grid
                const double t = block_sum(dot[k], red);
                if (threadIdx.x == 0) part[(size_t)k * nparts + blockIdx.x] = t;
            }
        }
    }
}

__global__ void __launch_bounds__(AT)
amgm_jacobi0_kernel(int32_t n, int K, const double* __restrict__ dinv, const double* __restrict__ b, double omega,
                    double* __restrict__ x) {
    ROW_LOOP(i, n) {
        const double d = omega * dinv[i];
        for (int k = 0; k < K; ++k) x[(int64_t)k * n + i] = d * b[(int64_t)k * n + i];
    }
}

__global__ void __launch_bounds__(AT)
amgm_restrict_kernel(int32_t n, int32_t nc, int K, const int32_t* __restrict__ pt_ptr, const int32_t* __restrict__ pt_idx,
                     const double* __restrict__ r, double* __restrict__ bc) {
    ROW_LOOP(I, nc) {
        const int32_t b0 = pt_ptr[I], e = pt_ptr[I + 1];
        for (int k = 0; k < K; ++k) {
            double s = 0.0;
            for (int32_t p = b0; p < e; ++p) s += r[(int64_t)k * n + pt_idx[p]];
            bc[(int64_t)k * nc + I] = s;
        }
    }
}

__global__ void __launch_bounds__(AT)
amgm_prolong_kernel(int32_t n, int32_t nc, int K, const int32_t* __restrict__ agg, const double* __restrict__ xc,
                    double scale, const double* __restrict__ x, double* __restrict__ xa) {
    ROW_LOOP(i, n) {
        const int32_t a = agg[i];
        for (int k = 0; k < K; ++k) xa[(int64_t)k * n + i] = x[(int64_t)k * n + i] + scale * xc[(int64_t)k * nc + a];
    }
}

// x_k = inv b_k, one warp per (row, k)
__global__ void __launch_bounds__(AT)
amgm_gemv_kernel(int32_t n, int K, const double* __restrict__ inv, const double* __restrict__ b, double* __restrict__ x) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t t = warp; t < (int64_t)n * K; t += nwarps) {
        const int64_t k = t / n, r = t - k * n;
        double acc = 0.0;
        for (int32_t j = lane; j < n; j += 32) acc = fma(inv[r * n + j], b[k * n + j], acc);
        acc = warp_sum(acc);
        if (lane == 0) x[k * n + r] = acc;
    }
}

// per-block partials of a_k . b_k
__global__ void __launch_bounds__(AT)
amgm_dot_kernel(int32_t n, int K, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ part,
                int nparts) {
    __shared__ double red[33];
    for (int k = 0; k < K; ++k) {
        double t = 0.0;
        ROW_LOOP(i, n) t = fma(a[(int64_t)k * n + i], b[(int64_t)k * n + i], t);
        t = block_sum(t, red);
        if (threadIdx.x == 0) part[(size_t)k * nparts + blockIdx.x] = t;
    }
}

// out[k] = sum of partial array k
__global__ void __launch_bounds__(AT)
amgm_sum_kernel(const double* __restrict__ part, int count, int nparts, int K, double* __restrict__ out) {
    __shared__ double red[33];
    for (int k = 0; k < K; ++k) {
        const double t = reduce_partials(part + (size_t)k * nparts, count, red);
        if (threadIdx.x == 0) out[k] = t;
    }
}

// alpha_k = rz_k / p_k.q_k ; x += alpha p ; r -= alpha q ; partials of r.r   (frozen systems untouched)
__global__ void __launch_bounds__(AT)
amgm_update_kernel(int32_t n, int K, const double* __restrict__ part_pq, int npq, int nparts, const double* __restrict__ rz,
                   const int* __restrict__ active, const double* __restrict__ p, const double* __restrict__ q,
                   double* __restrict__ x, double* __restrict__ r, double* __restrict__ part_rr) {
    __shared__ double red[33];
    for (int k = 0; k < K; ++k) {
        const double pq = reduce_partials(part_pq + (size_t)k * nparts, npq, red);
        const bool on = active[k] != 0;
        const double alpha = on ? rz[k] / pq : 0.0;
        double t = 0.0;
        ROW_LOOP(i, n) {
            const int64_t o = (int64_t)k * n + i;
            double ri = r[o];
            if (on) {
                x[o] = fma(alpha, p[o], x[o]);
                ri = fma(-alpha, q[o], ri);
                r[o] = ri;
            }
            t = fma(ri, ri, t);
        }
        t = block_sum(t, red);
        if (threadIdx.x == 0) part_rr[(size_t)k * nparts + blockIdx.x] = t;
    }
}

// rz'_k = r_k.z_k (from partials) ; beta = rz'/rz ; p = z + beta p
__global__ void __launch_bounds__(AT)
amgm_direction_kernel(int32_t n, int K, const double* __restrict__ part_rz, int nrz, int nparts,
                      const double* __restrict__ rz_old, double* __restrict__ rz_new, const int* __restrict__ active,
                      const double* __restrict__ z, double* __restrict__ p, int first) {
    __shared__ double red[33];
    for (int k = 0; k < K; ++k) {
        const double rzn = reduce_partials(part_rz + (size_t)k * nparts, nrz, red);
        const bool on = active[k] != 0;
        const double beta = first ? 0.0 : rzn / rz_old[k];
        if (on) {
            ROW_LOOP(i, n) {
                const int64_t o = (int64_t)k * n + i;
                p[o] = first ? z[o] : fma(beta, p[o], z[o]);
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) rz_new[k] = on ? rzn : rz_old[k];
    }
}

struct Work {
    std::vector<double*> x, r, b;      // per level: K * n_l doubles
    double *p = nullptr, *q = nullptr, *rr = nullptr, *z = nullptr, *part = nullptr, *scal = nullptr;
    int* active = nullptr;
    std::vector<void*> owned;
};

template <int MODE>
int sweep(const nodal_amg* h, const AmgLevel& V, int K, const double* b, const double* x, double* y, double* part,
          int nparts, cudaStream_t st) {
    const nodal_sell* m = V.sell;
    sell_launch(m, [&](auto a) {
        amgm_sell_kernel<MODE><<<amg_sell_grid(h->ctx, m->nslices), AT, 0, st>>>(
            m->n, m->nslices, m->slice_w, a, m->dinv, b, x, h->omega, y, part, K, nparts);
    });
    KERNEL_CHECK();
    return NODAL_OK;
}

// z_k = M b_k for the K vectors of a batch
int cycle_multi(const nodal_amg* h, Work& W, int K, const double* b0, double* z0, cudaStream_t st) {
    const nodal_ctx* ctx = h->ctx;
    const int last = (int)h->lv.size() - 1;
    for (int l = 0; l < last; ++l) {
        const AmgLevel& V = h->lv[l];
        const double* b = l == 0 ? b0 : W.b[l];
        amgm_jacobi0_kernel<<<amg_rows_grid(ctx, V.n), AT, 0, st>>>(V.n, K, V.sell->dinv, b, h->omega, W.x[l]);
        KERNEL_CHECK();
        NODAL_TRY(sweep<1>(h, V, K, b, W.x[l], W.r[l], nullptr, 0, st));
        amgm_restrict_kernel<<<amg_rows_grid(ctx, V.nc), AT, 0, st>>>(V.n, V.nc, K, V.pt_ptr, V.pt_idx, W.r[l], W.b[l + 1]);
        KERNEL_CHECK();
    }
    {
        const AmgLevel& V = h->lv[last];
        const double* b = last == 0 ? b0 : W.b[last];
        double* x = last == 0 ? z0 : W.x[last];
        if (h->inv) amgm_gemv_kernel<<<amg_rows_grid(ctx, (int64_t)V.n * 32 * K), AT, 0, st>>>(V.n, K, h->inv, b, x);
        else amgm_jacobi0_kernel<<<amg_rows_grid(ctx, V.n), AT, 0, st>>>(V.n, K, V.sell->dinv, b, h->omega, x);
        KERNEL_CHECK();
    }
    for (int l = last - 1; l >= 0; --l) {
        const AmgLevel& V = h->lv[l];
        const double* b = l == 0 ? b0 : W.b[l];
        double* xa = W.r[l];
        amgm_prolong_kernel<<<amg_rows_grid(ctx, V.n), AT, 0, st>>>(V.n, V.nc, K, V.agg, W.x[l + 1], h->scale, W.x[l], xa);
        KERNEL_CHECK();
        NODAL_TRY(sweep<2>(h, V, K, b, xa, l == 0 ? z0 : W.x[l], nullptr, 0, st));
    }
    return NODAL_OK;
}

}  // namespace

// rhs and x: K vectors of n doubles each, one after the other (x holds the initial guesses).
// iters_h / relres_h / status_h: K entries.  Returns NODAL_OK when every system converged, else the
// worst status (per-system ones in status_h).  K <= 8 per call.
extern "C" int nodal_amg_pcg_multi(nodal_ctx* ctx, nodal_amg* h, int32_t K, const double* rhs, double* x, double rtol,
                                   int32_t maxit, int32_t* iters_h, double* relres_h, int32_t* status_h, void* stream) {
    if (!ctx || !h || h->ctx != ctx || K < 1 || K > MK || !iters_h || !relres_h || !status_h) return NODAL_BAD_ARG;
    NvtxRange nvtx_range("nodal_amg_pcg_multi");
    for (int k = 0; k < K; ++k) { iters_h[k] = 0; relres_h[k] = 0.0; status_h[k] = NODAL_OK; }
    if (h->lv.empty()) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const AmgLevel& A = h->lv[0];
    const int32_t n = A.n;
    const int gv = amg_rows_grid(ctx, n), gs = amg_sell_grid(ctx, A.sell->nslices);
    const int nparts = std::max(gv, gs);
    Work W;
    auto alloc = [&](size_t count) -> double* {
        double* p = amg_pool<double>(ctx, count);
        if (p) W.owned.push_back(p);
        return p;
    };
    auto run = [&]() -> int {
        const int L = (int)h->lv.size();
        W.x.assign(L, nullptr); W.r.assign(L, nullptr); W.b.assign(L, nullptr);
        for (int l = 0; l < L; ++l) {
            const size_t len = (size_t)K * h->lv[l].n + 2;
            W.x[l] = alloc(len);
            W.r[l] = alloc(len);
            if (l > 0) W.b[l] = alloc(len);
            if (!W.x[l] || !W.r[l] || (l > 0 && !W.b[l])) return NODAL_CUDA_ERROR;
        }
        const size_t vlen = (size_t)K * n + 2;
        W.p = alloc(vlen); W.q = alloc(vlen); W.rr = alloc(vlen); W.z = alloc(vlen);
        W.part = alloc(3 * (size_t)MK * nparts + 8);
        W.scal = alloc(4 * MK + 8);
        W.active = reinterpret_cast<int*>(alloc(MK));
        if (!W.p || !W.q || !W.rr || !W.z || !W.part || !W.scal || !W.active) return NODAL_CUDA_ERROR;
        double* part_pq = W.part;
        double* part_rr = W.part + (size_t)MK * nparts;
        double* part_rz = W.part + 2 * (size_t)MK * nparts;
        double* rz[2] = {W.scal, W.scal + MK};
        double* norms = W.scal + 2 * MK;
        double* host = reinterpret_cast<double*>(static_cast<char*>(ctx->pinned) + 2048);   // MK doubles + MK ints
        int* host_active = reinterpret_cast<int*>(host + MK);

        auto norms_to_host = [&](const double* a, const double* b, double* out) -> int {
            amgm_dot_kernel<<<gv, AT, 0, st>>>(n, K, a, b, part_rr, nparts);
            KERNEL_CHECK();
            amgm_sum_kernel<<<1, AT, 0, st>>>(part_rr, gv, nparts, K, norms);
            KERNEL_CHECK();
            CUDA_TRY(cudaMemcpyAsync(host, norms, sizeof(double) * K, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            for (int k = 0; k < K; ++k) out[k] = host[k];
            return NODAL_OK;
        };
        double bb[MK], rrv[MK], bnorm[MK];
        int active[MK], iters[MK];
        NODAL_TRY(norms_to_host(rhs, rhs, bb));
        NODAL_TRY(sweep<1>(h, A, K, rhs, x, W.rr, nullptr, 0, st));      // r = b - A x0
        NODAL_TRY(norms_to_host(W.rr, W.rr, rrv));
        int remaining = 0;
        for (int k = 0; k < K; ++k) {
            iters[k] = 0;
            bnorm[k] = sqrt(bb[k]);
            if (!(bb[k] > 0.0)) {                       // b = 0 (x = 0 is the answer) or not finite
                active[k] = 0;
                status_h[k] = bb[k] == 0.0 ? NODAL_OK : NODAL_BREAKDOWN;
                relres_h[k] = 0.0;
                if (bb[k] == 0.0) CUDA_TRY(cudaMemsetAsync(x + (size_t)k * n, 0, sizeof(double) * (size_t)n, st));
                continue;
            }
            relres_h[k] = sqrt(rrv[k]) / bnorm[k];
            active[k] = relres_h[k] > rtol ? 1 : 0;
            remaining += active[k];
        }
        auto push_active = [&]() -> int {
            for (int k = 0; k < MK; ++k) host_active[k] = k < K ? active[k] : 0;
            CUDA_TRY(cudaMemcpyAsync(W.active, host_active, sizeof(int) * MK, cudaMemcpyHostToDevice, st));
            return NODAL_OK;
        };
        if (remaining) {
            NODAL_TRY(push_active());
            int par = 0;
            NODAL_TRY(cycle_multi(h, W, K, W.rr, W.z, st));
            amgm_dot_kernel<<<gv, AT, 0, st>>>(n, K, W.rr, W.z, part_rz, nparts);
            KERNEL_CHECK();
            amgm_direction_kernel<<<gv, AT, 0, st>>>(n, K, part_rz, gv, nparts, rz[par ^ 1], rz[par], W.active, W.z, W.p, 1);
            KERNEL_CHECK();
            for (int it = 0; it < maxit && remaining; ++it) {
                NODAL_TRY(sweep<0>(h, A, K, nullptr, W.p, W.q, part_pq, nparts, st));
                amgm_update_kernel<<<gv, AT, 0, st>>>(n, K, part_pq, gs, nparts, rz[par], W.active, W.p, W.q, x, W.rr, part_rr);
                KERNEL_CHECK();
                amgm_sum_kernel<<<1, AT, 0, st>>>(part_rr, gv, nparts, K, norms);
                KERNEL_CHECK();
                CUDA_TRY(cudaMemcpyAsync(host, norms, sizeof(double) * K, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                bool changed = false;
                for (int k = 0; k < K; ++k) {
                    if (!active[k]) continue;
                    ++iters[k];
                    const double rr = host[k];
                    if (!std::isfinite(rr)) { active[k] = 0; status_h[k] = NODAL_BREAKDOWN; changed = true; --remaining; continue; }
                    relres_h[k] = sqrt(rr) / bnorm[k];
                    // (a little inside the tolerance: there is no restart here, the true residual is checked once at the end)
                    if (relres_h[k] <= 0.7 * rtol) { active[k] = 0; changed = true; --remaining; }
                }
                if (!remaining) break;
                if (changed) NODAL_TRY(push_active());
                NODAL_TRY(cycle_multi(h, W, K, W.rr, W.z, st));
                amgm_dot_kernel<<<gv, AT, 0, st>>>(n, K, W.rr, W.z, part_rz, nparts);
                KERNEL_CHECK();
                amgm_direction_kernel<<<gv, AT, 0, st>>>(n, K, part_rz, gv, nparts, rz[par], rz[par ^ 1], W.active, W.z, W.p, 0);
                KERNEL_CHECK();
                par ^= 1;
            }
        }
        // true residuals
        NODAL_TRY(sweep<1>(h, A, K, rhs, x, W.rr, nullptr, 0, st));
        NODAL_TRY(norms_to_host(W.rr, W.rr, rrv));
        for (int k = 0; k < K; ++k) {
            iters_h[k] = iters[k];
            if (!(bb[k] > 0.0)) continue;
            relres_h[k] = sqrt(rrv[k]) / bnorm[k];
            if (status_h[k] == NODAL_OK && !(relres_h[k] <= rtol)) status_h[k] = NODAL_NOT_CONVERGED;
        }
        return NODAL_OK;
    };
    const int rc = run();
    cudaStreamSynchronize(st);
    for (void* p : W.owned) ctx_pool_free(ctx, p);
    if (rc != NODAL_OK) return rc;
    int worst = NODAL_OK;
    for (int k = 0; k < K; ++k) worst = std::max(worst, (int)status_h[k]);
    return worst;
}
