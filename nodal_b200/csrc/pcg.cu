// Jacobi-preconditioned conjugate gradients in FP64 -- replaces scipy's spsolve
// (nodal/nodal.py:325) for symmetric positive definite (R / A only) netlists.
//
// One CG iteration is three kernels, all persistent-grid and bandwidth bound:
//   K1 spmv_dot   q = A p,  partial sums of p.q                      (12 nnz + 20 n bytes)
//   K2 update     alpha = rz/pq ; x += alpha p ; r -= alpha q ;
//                 partial sums of r.D^-1 r and r.r                   (56 n bytes)
//   K3 direction  beta = rz'/rz ; p = D^-1 r + beta p                (32 n bytes)
// No scalar ever visits the host inside the loop: every block re-reduces the previous
// kernel's per-block partials in a fixed order (deterministic, bit-identical in all
// blocks), so alpha / beta / the convergence test are evaluated redundantly on device.
// Partials are double-buffered by iteration parity, which is baked into the kernel
// arguments of an (even, odd) iteration pair; CHUNK iterations are captured in one CUDA
// graph and the host only polls a `done` word between graph launches (two launches in
// flight, so the GPU never idles).  After `done`, the remaining kernels of a graph exit
// at their first instruction.
#include <algorithm>


#include "pcg_kernels.cuh"

constexpr int PCG_G2_PER_SM = 5;   // CTAs per SM of the vector kernels (measured best)

// ---------------------------------------------------------------- driver

extern "C" int nodal_pcg(nodal_ctx* ctx, int32_t n, int64_t nnz, const int32_t* indptr,
                         const int32_t* indices, const double* data, const double* rhs, double* x,
                         double rtol, int32_t maxit, int32_t flags, int32_t* iters_h,
                         double* relres_h, double* stats_h, void* stream) {
    NvtxRange nvtx_range("nodal_pcg");
    if (!ctx || n < 0 || !iters_h || !relres_h) return NODAL_BAD_ARG;
    *iters_h = 0;
    *relres_h = 0.0;
    if (stats_h) memset(stats_h, 0, 16 * sizeof(double));
    if (n == 0) return NODAL_OK;
    if (((uintptr_t)x & 15) || ((uintptr_t)rhs & 15)) {
        nodal_set_error("nodal_pcg: x and rhs must be 16-byte aligned");
        return NODAL_BAD_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaEvent_t ev_t0, ev_t1, ev_t2, ev_poll[2];
    CUDA_TRY(cudaEventCreate(&ev_t0));
    CUDA_TRY(cudaEventCreate(&ev_t1));
    CUDA_TRY(cudaEventCreate(&ev_t2));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[0], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_poll[1], cudaEventDisableTiming));
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t gexec = nullptr;
    cudaStream_t cap = nullptr;
    nodal_sell* sell = nullptr;
    int rc = NODAL_OK;
    int restarts = 0;
    PcgDev host{};
    float ms_setup = 0.f, ms_solve = 0.f;
    std::vector<cudaEvent_t> prof_ev;
    double prof_ms[4] = {0, 0, 0, 0};
    double* sc = nullptr;            // scale factors (pool)
    double un_rr = 0.0, un_bb = 0.0;
    // everything below funnels through `finish` so the resources above are released
    auto run = [&]() -> int {
        CUDA_TRY(cudaEventRecord(ev_t0, st));
        Mat A;
        A.n = n; A.nnz = nnz; A.indptr = indptr; A.indices = indices; A.data = data;
        const double mean = (double)nnz / n;
        A.tpr = mean <= 2.5 ? 2 : mean <= 6.0 ? 4 : mean <= 12.0 ? 8 : mean <= 24.0 ? 16 : 32;
        const int g2 = (int)std::min<int64_t>((int64_t)ctx->num_sms * PCG_G2_PER_SM,
                                              std::max<int64_t>(1, ((n >> 1) + PCG_THREADS - 1) / PCG_THREADS));
        // symmetric diagonal scaling (only with the private SELL copy, only for positive diagonals)
        bool scaled = false;
        if (!(flags & NODAL_PCG_FORCE_CSR)) {
            if (!(flags & NODAL_PCG_NO_SCALE)) {
                sc = static_cast<double*>(ctx_pool_alloc(ctx, sizeof(double) * (size_t)n + 256));
                if (!sc) return NODAL_CUDA_ERROR;
                int* flag = reinterpret_cast<int*>(sc + n);
                CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
                pcg_scale_factors_kernel<<<g2, PCG_THREADS, 0, st>>>(n, indptr, indices, data, sc, flag);
                KERNEL_CHECK();
                int* flag_h = reinterpret_cast<int*>(ctx->pinned);
                CUDA_TRY(cudaMemcpyAsync(flag_h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                scaled = (*flag_h == 0);
            }
            NODAL_TRY(sell_from_csr(ctx, n, nnz, indptr, indices, data, &sell, st, scaled ? sc : nullptr));
            if ((double)sell->padded <= 1.5 * (double)nnz + 1024.0) A.sell = sell;
            else scaled = false;
        }
        if (A.sell) {
            const int64_t want = ((int64_t)sell->nslices * 32 + PCG_THREADS - 1) / PCG_THREADS;
            A.g1 = (int)std::min<int64_t>((int64_t)ctx->num_sms * PCG_SELL_CTAS_PER_SM, want);
        } else {
            const int64_t want = ((int64_t)n * A.tpr + PCG_THREADS - 1) / PCG_THREADS;
            A.g1 = (int)std::min<int64_t>((int64_t)ctx->num_sms * 8, want);
        }
        const size_t vec = align_up(sizeof(double) * (size_t)n, 256);
        const int gmax = std::max(A.g1, g2);
        const size_t partb = align_up(sizeof(double) * (size_t)gmax, 256);
        NODAL_TRY(ctx_reserve(ctx, 5 * vec + 8 * partb + 4096));
        double* r = carve<double>(ctx, n);
        double* bh = scaled ? carve<double>(ctx, n) : nullptr;   // S b
        double* p = carve<double>(ctx, n);
        double* q = carve<double>(ctx, n);
        double* dinv_own = nullptr;
        const double* dinv = nullptr;
        if (A.sell) dinv = sell->dinv;
        else {
            dinv_own = carve<double>(ctx, n);
            dinv = dinv_own;
        }
        double* part_pq[2] = {carve<double>(ctx, gmax), carve<double>(ctx, gmax)};
        double* part_rz[2] = {carve<double>(ctx, gmax), carve<double>(ctx, gmax)};
        double* part_rr[2] = {carve<double>(ctx, gmax), carve<double>(ctx, gmax)};
        double* part_bb = carve<double>(ctx, gmax);
        PcgDev* dev = carve<PcgDev>(ctx, 1);
        if (!r || !p || !q || !dinv || !part_bb || !dev) return NODAL_CUDA_ERROR;
        if (dinv_own) {
            csr_dinv_kernel<<<g2, PCG_THREADS, 0, st>>>(n, indptr, indices, data, dinv_own);
            KERNEL_CHECK();
        }
        CUDA_TRY(cudaMemsetAsync(dev, 0, sizeof(PcgDev), st));
        const double* b_eff = rhs;
        if (scaled) {
            if (!bh) return NODAL_CUDA_ERROR;
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(n, rhs, sc, bh, 0);     // b_hat = S b
            KERNEL_CHECK();
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(n, x, sc, x, 1);        // x_hat = S^-1 x0
            KERNEL_CHECK();
            b_eff = bh;
        }

        auto spmv_plain = [&](const double* in, double* out) -> int {
            if (A.sell) return nodal_sell_spmv(ctx, A.sell, in, out, st);
            return csr_spmv_launch(ctx, n, nnz, indptr, indices, data, in, out, st);
        };
        auto start = [&](int first) -> int {  // (re)start from the current x
            NODAL_TRY(spmv_plain(x, q));
            if (scaled)
                pcg_start_kernel<true><<<g2, PCG_THREADS, 0, st>>>(n, b_eff, q, dinv, r, p, part_rz[1],
                                                                   part_rr[1], part_bb);
            else
                pcg_start_kernel<false><<<g2, PCG_THREADS, 0, st>>>(n, b_eff, q, dinv, r, p, part_rz[1],
                                                                    part_rr[1], part_bb);
            KERNEL_CHECK();
            pcg_scalars_kernel<<<1, PCG_THREADS, 0, st>>>(dev, part_rr[1], part_bb, g2, rtol, maxit,
                                                          first);
            KERNEL_CHECK();
            return NODAL_OK;
        };
        auto launch_k2 = [&](int par, cudaStream_t s) -> int {
            if (scaled)
                pcg_update_kernel<true><<<g2, PCG_THREADS, 0, s>>>(dev, n, part_pq[par], A.g1, part_rz[par ^ 1], g2,
                                                                   x, p, r, q, dinv, part_rz[par], part_rr[par]);
            else
                pcg_update_kernel<false><<<g2, PCG_THREADS, 0, s>>>(dev, n, part_pq[par], A.g1, part_rz[par ^ 1], g2,
                                                                    x, p, r, q, dinv, part_rz[par], part_rr[par]);
            KERNEL_CHECK();
            return NODAL_OK;
        };
        auto launch_k3 = [&](int par, cudaStream_t s) -> int {
            if (scaled)
                pcg_direction_kernel<true><<<g2, PCG_THREADS, 0, s>>>(dev, n, part_rz[par ^ 1], part_rz[par],
                                                                      part_rr[par], g2, p, r, dinv);
            else
                pcg_direction_kernel<false><<<g2, PCG_THREADS, 0, s>>>(dev, n, part_rz[par ^ 1], part_rz[par],
                                                                       part_rr[par], g2, p, r, dinv);
            KERNEL_CHECK();
            return NODAL_OK;
        };
        auto iteration = [&](int par, cudaStream_t s) -> int {
            NODAL_TRY(launch_k1(A, dev, p, q, part_pq[par], s));
            NODAL_TRY(launch_k2(par, s));
            NODAL_TRY(launch_k3(par, s));
            return NODAL_OK;
        };

        const bool profile = (flags & NODAL_PCG_PROFILE) != 0;
        const bool use_graph = !(flags & NODAL_PCG_NO_GRAPH) && !profile;
        if (profile) {
            prof_ev.resize(PCG_CHUNK * 4);
            for (auto& e : prof_ev) CUDA_TRY(cudaEventCreate(&e));
        }
        if (use_graph) {
            const unsigned long long before = g_nodal_launches;
            CUDA_TRY(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
            CUDA_TRY(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
            int crc = NODAL_OK;
            for (int i = 0; i < PCG_CHUNK && crc == NODAL_OK; ++i) crc = iteration(i & 1, cap);
            cudaError_t ce = cudaStreamEndCapture(cap, &graph);
            if (crc != NODAL_OK) return crc;
            CUDA_TRY(ce);
            CUDA_TRY(cudaGraphInstantiate(&gexec, graph, 0));
            g_nodal_launches = before;  // captured nodes are counted per graph launch below
        }
        NODAL_TRY(start(1));
        CUDA_TRY(cudaEventRecord(ev_t1, st));

        PcgDev* poll = reinterpret_cast<PcgDev*>(ctx->pinned);  // two slots
        double last_true_rr = -1.0;
        for (;;) {
            // run chunks until the device reports done
            const int64_t max_chunks = (int64_t)maxit / PCG_CHUNK + 3;
            int64_t k = 0;
            for (;; ++k) {
                if (use_graph) {
                    CUDA_TRY(cudaGraphLaunch(gexec, st));
                    g_nodal_launches += 3ull * PCG_CHUNK;
                } else if (profile) {
                    const int it0 = host.iters;
                    for (int i = 0; i < PCG_CHUNK; ++i) {
                        const int par = i & 1;
                        CUDA_TRY(cudaEventRecord(prof_ev[4 * i + 0], st));
                        NODAL_TRY(launch_k1(A, dev, p, q, part_pq[par], st));
                        CUDA_TRY(cudaEventRecord(prof_ev[4 * i + 1], st));
                        NODAL_TRY(launch_k2(par, st));
                        CUDA_TRY(cudaEventRecord(prof_ev[4 * i + 2], st));
                        NODAL_TRY(launch_k3(par, st));
                        CUDA_TRY(cudaEventRecord(prof_ev[4 * i + 3], st));
                    }
                    CUDA_TRY(cudaMemcpyAsync(&poll[0], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                    const int ran = poll[0].iters - it0;  // iterations that did real work
                    for (int i = 0; i < ran && i < PCG_CHUNK; ++i) {
                        float a = 0, b = 0, c = 0;
                        CUDA_TRY(cudaEventElapsedTime(&a, prof_ev[4 * i + 0], prof_ev[4 * i + 1]));
                        CUDA_TRY(cudaEventElapsedTime(&b, prof_ev[4 * i + 1], prof_ev[4 * i + 2]));
                        CUDA_TRY(cudaEventElapsedTime(&c, prof_ev[4 * i + 2], prof_ev[4 * i + 3]));
                        prof_ms[0] += a; prof_ms[1] += b; prof_ms[2] += c; prof_ms[3] += 1.0;
                    }
                    host = poll[0];
                } else {
                    for (int i = 0; i < PCG_CHUNK; ++i) NODAL_TRY(iteration(i & 1, st));
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
            if (!host.done) { host.status = NODAL_NOT_CONVERGED; }
            if (host.status == NODAL_BREAKDOWN) break;
            // true residual of the returned x
            NODAL_TRY(start(0));
            CUDA_TRY(cudaMemcpyAsync(&poll[0], dev, sizeof(PcgDev), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            const int recurrence_status = host.status;
            host = poll[0];
            if (scaled) {
                // the contract is on the UNSCALED residual: ||b - A x|| <= rtol ||b||
                pcg_unscaled_norm_kernel<<<g2, PCG_THREADS, 0, st>>>(n, r, sc, rhs, part_rr[0], part_bb);
                KERNEL_CHECK();
                std::vector<double> hp(2 * (size_t)g2);
                CUDA_TRY(cudaMemcpyAsync(hp.data(), part_rr[0], sizeof(double) * g2, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaMemcpyAsync(hp.data() + g2, part_bb, sizeof(double) * g2, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                double rr_un = 0.0, bb_un = 0.0;
                for (int i = 0; i < g2; ++i) { rr_un += hp[i]; bb_un += hp[g2 + i]; }
                un_rr = rr_un; un_bb = bb_un;
                const double target = rtol * rtol * bb_un;
                if (host.rr <= host.tol2 && rr_un > target && recurrence_status == NODAL_OK &&
                    host.iters < host.maxit && restarts < 8) {
                    // converged in the scaled norm only: tighten the scaled threshold and go on
                    const double tol2 = host.tol2 * std::min(0.25, 0.25 * target / rr_un);
                    const int zero = 0;
                    CUDA_TRY(cudaMemcpyAsync(&dev->tol2, &tol2, sizeof(double), cudaMemcpyHostToDevice, st));
                    CUDA_TRY(cudaMemcpyAsync(&dev->done, &zero, sizeof(int), cudaMemcpyHostToDevice, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                    ++restarts;
                    continue;
                }
                if (rr_un <= target) { host.status = NODAL_OK; break; }
                if (host.rr <= host.tol2) { host.status = NODAL_NOT_CONVERGED; break; }
            }
            if (host.rr <= host.tol2) { host.status = NODAL_OK; break; }
            if (recurrence_status == NODAL_NOT_CONVERGED || host.iters >= host.maxit) {
                host.status = NODAL_NOT_CONVERGED;
                break;
            }
            // recurrence said converged but the true residual is above tolerance: restart
            if (restarts >= 8 || (last_true_rr >= 0.0 && host.rr > 0.25 * last_true_rr)) {
                host.status = NODAL_NOT_CONVERGED;  // attainable accuracy reached
                break;
            }
            last_true_rr = host.rr;
            ++restarts;
        }
        CUDA_TRY(cudaEventRecord(ev_t2, st));
        CUDA_TRY(cudaEventSynchronize(ev_t2));
        CUDA_TRY(cudaEventElapsedTime(&ms_setup, ev_t0, ev_t1));
        CUDA_TRY(cudaEventElapsedTime(&ms_solve, ev_t1, ev_t2));
        if (scaled) {
            pcg_scale_vec_kernel<<<g2, PCG_THREADS, 0, st>>>(n, x, sc, x, 0);        // x = S x_hat
            KERNEL_CHECK();
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        *iters_h = host.iters;
        *relres_h = host.bb > 0.0 ? sqrt(host.rr / host.bb) : 0.0;
        if (scaled && un_bb > 0.0) *relres_h = sqrt(un_rr / un_bb);
        if (stats_h) {
            stats_h[0] = host.iters;
            stats_h[1] = *relres_h;
            stats_h[2] = restarts;
            stats_h[3] = ms_solve;
            stats_h[4] = ms_setup;
            stats_h[5] = A.sell ? 1.0 : 0.0;
            stats_h[6] = A.sell ? (double)sell->padded : (double)nnz;
            stats_h[7] = A.g1;
            stats_h[12] = scaled ? 1.0 : 0.0;
            if (prof_ms[3] > 0) {
                stats_h[8] = prof_ms[0] / prof_ms[3];
                stats_h[9] = prof_ms[1] / prof_ms[3];
                stats_h[10] = prof_ms[2] / prof_ms[3];
                stats_h[11] = prof_ms[3];
            }
        }
        return host.status;
    };
    rc = run();
    if (gexec) cudaGraphExecDestroy(gexec);
    if (graph) cudaGraphDestroy(graph);
    if (cap) cudaStreamDestroy(cap);
    for (auto& e : prof_ev) cudaEventDestroy(e);
    if (sell) { cudaStreamSynchronize(st); sell_free(sell); }
    if (sc) ctx_pool_free(ctx, sc);
    cudaEventDestroy(ev_t0); cudaEventDestroy(ev_t1); cudaEventDestroy(ev_t2);
    cudaEventDestroy(ev_poll[0]); cudaEventDestroy(ev_poll[1]);
    return rc;
}
