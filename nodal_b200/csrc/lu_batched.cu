// Batched small-system solve for parameter sweeps (config C4): every thread stamps its own
// copy of a shared topology from its row of `values` and solves the n x n system with
// partially pivoted Gaussian elimination.  The matrix never touches HBM: it lives in
// shared memory, element-major / thread-minor so that all lanes of a warp hit different
// banks.  Algorithmic traffic is ncomp + n doubles per system.
// Replaces a Python loop of Netlist + Circuit + numpy.linalg.solve (nodal/nodal.py:306-336).
#include <algorithm>
#include <utility>

#include "common.cuh"
#include "stamp_core.cuh"

constexpr int BATCH_MAX_N = 24;

__global__ void lu_batched_kernel(int64_t batch, int ncomp, const uint8_t* __restrict__ type,
                                  const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                                  const int32_t* __restrict__ c, const int32_t* __restrict__ d,
                                  const int32_t* __restrict__ drv, const int32_t* __restrict__ branch,
                                  int kcl, int n, const double* __restrict__ values,
                                  double* __restrict__ x, int32_t* __restrict__ info) {
    extern __shared__ double M[];   // [(n) * (n + 1)][blockDim.x]
    const int T = blockDim.x, tid = threadIdx.x;
    const int ld = n + 1;
#define AT(i, j) M[((i) * ld + (j)) * T + tid]
    for (int64_t sys = (int64_t)blockIdx.x * T + tid; sys < batch; sys += (int64_t)gridDim.x * T) {
        for (int e = 0; e < n * ld; ++e) M[e * T + tid] = 0.0;
        const double* val = values + sys * ncomp;
        for (int k = 0; k < ncomp; ++k) {
            const int t = type[k];
            double dv = 1.0;
            if ((t == NODAL_T_CCVS || t == NODAL_T_CCCS) && drv) dv = val[drv[k]];
            StampOut o;    // c / d / drv / branch may be null for R / A-only topologies
            stamp_component(t, val[k], a[k], b[k], c ? c[k] : -2, d ? d[k] : -2, dv, branch ? branch[k] : -1, kcl, n, o);
            for (int e = 0; e < o.count; ++e) AT(o.row[e], o.col[e]) += o.val[e];   // col == n is the rhs
        }
        int bad = 0;
        for (int k = 0; k < n && !bad; ++k) {
            int p = k;
            double best = fabs(AT(k, k));
            for (int i = k + 1; i < n; ++i) {
                const double v = fabs(AT(i, k));
                if (v > best) { best = v; p = i; }
            }
            if (!(best > 0.0)) { bad = k + 1; break; }
            if (p != k)
                for (int j = k; j <= n; ++j) { const double t0 = AT(k, j); AT(k, j) = AT(p, j); AT(p, j) = t0; }
            const double inv = 1.0 / AT(k, k);
            for (int i = k + 1; i < n; ++i) {
                const double l = AT(i, k) * inv;
                if (l != 0.0)
                    for (int j = k + 1; j <= n; ++j) AT(i, j) = fma(-l, AT(k, j), AT(i, j));
            }
        }
        double* xs = x + sys * n;
        if (bad) {
            for (int i = 0; i < n; ++i) xs[i] = nan("");
        } else {
            for (int i = n - 1; i >= 0; --i) {
                double s = AT(i, n);
                for (int j = i + 1; j < n; ++j) s = fma(-AT(i, j), AT(j, n), s);
                s /= AT(i, i);
                AT(i, n) = s;
                xs[i] = s;
            }
        }
        info[sys] = bad;
    }
#undef AT
}

// Register-resident variant for small systems (n <= 8, the op-amp sweeps of config C4 have n = 6):
// the stamping still scatters into the thread's shared-memory column (row / column of an emitted
// entry are run-time values), then the n x (n + 1) augmented matrix moves into registers and the
// whole elimination runs on statically indexed registers -- independent FMA chains instead of
// ~600 dependent shared-memory round trips per system.  Same operations in the same order as the
// generic kernel (results are bit-identical).  SOA: values are [ncomp][batch] and x is [n][batch]
// (every load / store of a warp is one contiguous 256-byte request) instead of [batch][ncomp] /
// [batch][n].
// Compile-time loops: nvcc keeps the n x (n + 1) array in local memory when the triangular loops
// are only `#pragma unroll`ed (336-byte stack frame, ~780 local loads / stores); with the indices
// as template constants every element is a register.
template <int... I, typename F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, I...>, F&& f) {
    (f(std::integral_constant<int, I>{}), ...);
}
template <int COUNT, typename F>
__device__ __forceinline__ void static_for(F&& f) {
    static_for_impl(std::make_integer_sequence<int, (COUNT > 0 ? COUNT : 0)>{}, static_cast<F&&>(f));
}

template <int N, bool SOA>
__global__ void __launch_bounds__(128)
lu_batched_reg_kernel(int64_t batch, int ncomp, const uint8_t* __restrict__ type,
                      const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                      const int32_t* __restrict__ c, const int32_t* __restrict__ d,
                      const int32_t* __restrict__ drv, const int32_t* __restrict__ branch,
                      int kcl, const double* __restrict__ values, double* __restrict__ x,
                      int32_t* __restrict__ info) {
    extern __shared__ double M[];   // [N * (N + 1)][blockDim.x]
    const int T = blockDim.x, tid = threadIdx.x;
    constexpr int LD = N + 1;
    for (int64_t sys = (int64_t)blockIdx.x * T + tid; sys < batch; sys += (int64_t)gridDim.x * T) {
#pragma unroll
        for (int e = 0; e < N * LD; ++e) M[e * T + tid] = 0.0;
        const double* val = SOA ? values + sys : values + sys * ncomp;
        const int64_t vs = SOA ? batch : 1;
        for (int k = 0; k < ncomp; ++k) {
            const int t = type[k];
            double dv = 1.0;
            if ((t == NODAL_T_CCVS || t == NODAL_T_CCCS) && drv) dv = val[(int64_t)drv[k] * vs];
            StampOut o;
            stamp_component(t, val[(int64_t)k * vs], a[k], b[k], c ? c[k] : -2, d ? d[k] : -2, dv,
                            branch ? branch[k] : -1, kcl, N, o);
            static_for<6>([&](auto E) {          // a component emits at most 6 entries (stamp_core.cuh)
                constexpr int e = E;
                if (e < o.count) M[(o.row[e] * LD + o.col[e]) * T + tid] += o.val[e];   // col == N is the rhs
            });
        }
        double A[N][LD];
        static_for<N>([&](auto I) { static_for<LD>([&](auto J) { A[I][J] = M[(I * LD + J) * T + tid]; }); });
        int bad = 0;
        static_for<N>([&](auto K) {
            constexpr int k = K;
            int p = k;
            double best = fabs(A[k][k]);
            static_for<N - 1 - k>([&](auto D) {
                constexpr int i = k + 1 + D;
                const double v = fabs(A[i][k]);
                if (v > best) { best = v; p = i; }
            });
            if (!(best > 0.0) && !bad) bad = k + 1;
            static_for<N - 1 - k>([&](auto D) {
                constexpr int i = k + 1 + D;
                const bool sw = (p == i);
                static_for<LD - k>([&](auto E) {
                    constexpr int j = k + E;
                    const double t0 = A[k][j], t1 = A[i][j];
                    A[k][j] = sw ? t1 : t0;
                    A[i][j] = sw ? t0 : t1;
                });
            });
            const double inv = 1.0 / A[k][k];
            static_for<N - 1 - k>([&](auto D) {
                constexpr int i = k + 1 + D;
                const double l = A[i][k] * inv;
                static_for<LD - 1 - k>([&](auto E) { constexpr int j = k + 1 + E; A[i][j] = fma(-l, A[k][j], A[i][j]); });
            });
        });
        static_for<N>([&](auto R) {
            constexpr int i = N - 1 - R;
            double s = A[i][N];
            static_for<N - 1 - i>([&](auto E) { constexpr int j = i + 1 + E; s = fma(-A[i][j], A[j][N], s); });
            s /= A[i][i];
            A[i][N] = s;
        });
        const double qnan = nan("");
        static_for<N>([&](auto I) {
            const double v = bad ? qnan : A[I][N];
            if (SOA) x[(int64_t)I * batch + sys] = v;
            else x[sys * N + I] = v;
        });
        info[sys] = bad;
    }
}

template <bool SOA>
static int launch_reg(nodal_ctx* ctx, int64_t batch, int32_t ncomp, const uint8_t* type, const int32_t* a,
                      const int32_t* b, const int32_t* c, const int32_t* d, const int32_t* drv,
                      const int32_t* branch, int32_t kcl, int32_t n, const double* values, double* x,
                      int32_t* info, cudaStream_t st) {
    const int threads = 128;
    const size_t smem = sizeof(double) * (size_t)n * (n + 1) * threads;
    const int64_t want = (batch + threads - 1) / threads;
    const int grid = (int)std::min<int64_t>(want, (int64_t)ctx->num_sms * 32);
#define REG_CASE(NN)                                                                                          \
    case NN:                                                                                                  \
        CUDA_TRY(cudaFuncSetAttribute(lu_batched_reg_kernel<NN, SOA>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      (int)smem));                                                            \
        lu_batched_reg_kernel<NN, SOA><<<grid, threads, smem, st>>>(batch, ncomp, type, a, b, c, d, drv, branch, \
                                                                    kcl, values, x, info);                    \
        break;
    switch (n) {
        REG_CASE(1) REG_CASE(2) REG_CASE(3) REG_CASE(4) REG_CASE(5) REG_CASE(6) REG_CASE(7) REG_CASE(8)
        default: return NODAL_BAD_ARG;
    }
#undef REG_CASE
    KERNEL_CHECK();
    return NODAL_OK;
}

extern "C" int nodal_lu_batched(nodal_ctx* ctx, int64_t batch, int32_t ncomp, const uint8_t* type,
                                const int32_t* a, const int32_t* b, const int32_t* c,
                                const int32_t* d, const int32_t* drv, const int32_t* branch,
                                int32_t kcl, int32_t n, const double* values, double* x,
                                int32_t* info, void* stream) {
    if (!ctx || batch < 0 || ncomp < 0 || n < 0) return NODAL_BAD_ARG;
    if (n > BATCH_MAX_N) {
        nodal_set_error("nodal_lu_batched: n=%d > %d unknowns per system is not supported", n, BATCH_MAX_N);
        return NODAL_BAD_ARG;
    }
    if (batch == 0 || n == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (n <= 8)
        return launch_reg<false>(ctx, batch, ncomp, type, a, b, c, d, drv, branch, kcl, n, values, x, info,
                                 (cudaStream_t)stream);
    const size_t per_thread = sizeof(double) * (size_t)n * (n + 1);
    int threads = (int)std::min<size_t>(128, (200 * 1024) / per_thread);
    threads = std::max(32, threads / 32 * 32);
    const size_t smem = per_thread * threads;
    CUDA_TRY(cudaFuncSetAttribute(lu_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t want = (batch + threads - 1) / threads;
    const int grid = (int)std::min<int64_t>(want, (int64_t)ctx->num_sms * 16);
    lu_batched_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(batch, ncomp, type, a, b, c, d, drv,
                                                                     branch, kcl, n, values, x, info);
    KERNEL_CHECK();
    return NODAL_OK;
}

// Transposed layout: values_t is [ncomp][batch], x_t is [n][batch] (system index fastest), so every
// parameter load and solution store of a warp is one contiguous request.  n <= 8.
extern "C" int nodal_lu_batched_soa(nodal_ctx* ctx, int64_t batch, int32_t ncomp, const uint8_t* type,
                                    const int32_t* a, const int32_t* b, const int32_t* c,
                                    const int32_t* d, const int32_t* drv, const int32_t* branch,
                                    int32_t kcl, int32_t n, const double* values_t, double* x_t,
                                    int32_t* info, void* stream) {
    if (!ctx || batch < 0 || ncomp < 0 || n < 0) return NODAL_BAD_ARG;
    if (n > 8) {
        nodal_set_error("nodal_lu_batched_soa: n=%d > 8 unknowns per system is not supported", n);
        return NODAL_BAD_ARG;
    }
    if (batch == 0 || n == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    return launch_reg<true>(ctx, batch, ncomp, type, a, b, c, d, drv, branch, kcl, n, values_t, x_t, info,
                            (cudaStream_t)stream);
}
