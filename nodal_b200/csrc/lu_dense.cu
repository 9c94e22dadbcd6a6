// Blocked FP64 LU with partial pivoting + triangular solves on a row-major n x n matrix.
// Replaces numpy.linalg.solve -> LAPACK dgesv (nodal/nodal.py:327).
//
// Right-looking, block size NB = 128.  Per block column k:
//   1. lu_panel_kernel      cooperative kernel: the (n-k) x NB panel is spread over up to one
//                           CTA per SM and kept in shared memory for all NB column steps;
//                           one grid-wide sync per column elects the pivot (max |a|, lowest
//                           row on ties, as LAPACK idamax) and broadcasts the pivot row.
//   2. lu_swap_rows_kernel  the panel's row interchanges applied to the columns left and
//                           right of the panel (dlaswp).
//   3. lu_trsm_kernel       U12 = L11^-1 A12, 64-column slabs solved in shared memory.
//   4. lu_gemm_kernel       A22 -= L21 U12 on the FP64 tensor pipe: mma.sync m8n8k4 DMMA,
//                           128x128 CTA tiles, cp.async double-buffered K chunks of 32.
// Then P b, forward and backward substitution in blocks of 128 (diagonal solve + GEMV).
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"

namespace cg = cooperative_groups;

constexpr int LU_NB = 128;
constexpr int PANEL_THREADS = 512;
constexpr int PANEL_LD = LU_NB + 1;

struct PivotCand {
    double absval;
    int row;
    int pad;
};

__device__ __forceinline__ bool better(double v, int r, double bv, int br) {
    return v > bv || (v == bv && r < br);
}

__global__ void __launch_bounds__(PANEL_THREADS, 1)
lu_panel_kernel(double* __restrict__ A, int n, int k, int jb, int rows_per_cta, int* __restrict__ ipiv,
                PivotCand* cand, double* candrow, double* diagrow, int* info) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ double smem[];
    double* tile = smem;                                   // [rows_per_cta][PANEL_LD]
    double* prow = tile + (size_t)rows_per_cta * PANEL_LD; // [LU_NB]
    __shared__ double s_val[32];
    __shared__ int s_row[32];
    __shared__ int s_cta[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = PANEL_THREADS / 32;
    const int ncta = gridDim.x;
    const int r0 = k + blockIdx.x * rows_per_cta;
    const int R = max(0, min(rows_per_cta, n - r0));

    for (int idx = tid; idx < R * jb; idx += PANEL_THREADS) {
        const int i = idx / jb, c = idx - i * jb;
        tile[i * PANEL_LD + c] = A[(size_t)(r0 + i) * n + k + c];
    }
    __syncthreads();

    for (int j = 0; j < jb; ++j) {
        const int g = k + j, par = j & 1;
        // ---- local pivot candidate
        double best = -1.0;
        int brow = 0x7fffffff;
        for (int i = tid; i < R; i += PANEL_THREADS) {
            const int gi = r0 + i;
            if (gi >= g) {
                const double v = fabs(tile[i * PANEL_LD + j]);
                if (better(v, gi, best, brow)) { best = v; brow = gi; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int orow = __shfl_xor_sync(0xffffffffu, brow, o);
            if (better(ov, orow, best, brow)) { best = ov; brow = orow; }
        }
        if (lane == 0) { s_val[warp] = best; s_row[warp] = brow; }
        __syncthreads();
        if (warp == 0) {
            best = lane < nwarps ? s_val[lane] : -1.0;
            brow = lane < nwarps ? s_row[lane] : 0x7fffffff;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                const int orow = __shfl_xor_sync(0xffffffffu, brow, o);
                if (better(ov, orow, best, brow)) { best = ov; brow = orow; }
            }
            if (lane == 0) { s_val[0] = best; s_row[0] = brow; }
        }
        __syncthreads();
        best = s_val[0];
        brow = s_row[0];
        // ---- publish candidate (+ its row) and the current diagonal row
        const size_t slot = (size_t)par * ncta + blockIdx.x;
        if (tid == 0) { cand[slot].absval = best; cand[slot].row = brow; }
        if (best >= 0.0) {
            const int li = brow - r0;
            for (int c = tid; c < jb; c += PANEL_THREADS) candrow[slot * LU_NB + c] = tile[li * PANEL_LD + c];
        }
        if (g >= r0 && g < r0 + R) {
            const int li = g - r0;
            for (int c = tid; c < jb; c += PANEL_THREADS) diagrow[(size_t)par * LU_NB + c] = tile[li * PANEL_LD + c];
        }
        __threadfence();
        grid.sync();
        // ---- elect the global pivot (all CTAs, identically)
        if (warp == 0) {
            double gv = -1.0;
            int gr = 0x7fffffff, gc = 0;
            for (int c = lane; c < ncta; c += 32) {
                const PivotCand* pc = &cand[(size_t)par * ncta + c];
                const double v = __ldcg(&pc->absval);
                const int r = __ldcg(&pc->row);
                if (better(v, r, gv, gr)) { gv = v; gr = r; gc = c; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, gv, o);
                const int orow = __shfl_xor_sync(0xffffffffu, gr, o);
                const int oc = __shfl_xor_sync(0xffffffffu, gc, o);
                if (better(ov, orow, gv, gr)) { gv = ov; gr = orow; gc = oc; }
            }
            if (lane == 0) { s_val[1] = gv; s_row[1] = gr; s_cta[1] = gc; }
        }
        __syncthreads();
        const double pv_abs = s_val[1];
        // No candidate at all (every entry at or below the diagonal is NaN: better() never picks
        // one): keep row g where it is -- the swap is a no-op, info is flagged below and the NaNs
        // propagate into the solution as LAPACK's do -- instead of electing row INT_MAX.
        const bool none = !(pv_abs >= 0.0);
        const int pv_row = none ? g : s_row[1], pv_cta = s_cta[1];
        for (int c = tid; c < jb; c += PANEL_THREADS)
            prow[c] = none ? __ldcg(&diagrow[(size_t)par * LU_NB + c])
                           : __ldcg(&candrow[((size_t)par * ncta + pv_cta) * LU_NB + c]);
        if (blockIdx.x == 0 && tid == 0) {
            ipiv[g] = pv_row;
            if (!(pv_abs > 0.0)) atomicCAS(info, 0, g + 1);   // exact zero (or NaN) pivot
        }
        // ---- row interchange inside the panel (both sources are the published copies)
        if (pv_row != g) {
            if (pv_row >= r0 && pv_row < r0 + R) {
                const int li = pv_row - r0;
                for (int c = tid; c < jb; c += PANEL_THREADS)
                    tile[li * PANEL_LD + c] = __ldcg(&diagrow[(size_t)par * LU_NB + c]);
            }
        }
        __syncthreads();   // prow complete
        if (pv_row != g && g >= r0 && g < r0 + R) {
            const int li = g - r0;
            for (int c = tid; c < jb; c += PANEL_THREADS) tile[li * PANEL_LD + c] = prow[c];
        }
        __syncthreads();
        // ---- eliminate column j below the diagonal
        const double piv = prow[j];
        if (piv != 0.0 && piv == piv) {
            const double inv = 1.0 / piv;
            for (int i = tid; i < R; i += PANEL_THREADS)
                if (r0 + i > g) tile[i * PANEL_LD + j] *= inv;
            __syncthreads();
            for (int i = warp; i < R; i += nwarps) {
                if (r0 + i <= g) continue;
                const double l = tile[i * PANEL_LD + j];
                for (int c = j + 1 + lane; c < jb; c += 32)
                    tile[i * PANEL_LD + c] = fma(-l, prow[c], tile[i * PANEL_LD + c]);
            }
        }
        __syncthreads();
    }
    for (int idx = tid; idx < R * jb; idx += PANEL_THREADS) {
        const int i = idx / jb, c = idx - i * jb;
        A[(size_t)(r0 + i) * n + k + c] = tile[i * PANEL_LD + c];
    }
}

// dlaswp on the columns [c_begin, c_end) (outside the panel): one thread per column, swaps applied in order.
__global__ void __launch_bounds__(256)
lu_swap_rows_kernel(double* __restrict__ A, int n, int k, int jb, const int* __restrict__ ipiv, int c_begin, int c_end) {
    for (int c = c_begin + blockIdx.x * blockDim.x + threadIdx.x; c < c_end; c += gridDim.x * blockDim.x) {
        for (int j = 0; j < jb; ++j) {
            const int r1 = k + j, r2 = ipiv[r1];
            if (r2 != r1 && r2 >= 0 && r2 < n) {
                const double a = A[(size_t)r1 * n + c], b = A[(size_t)r2 * n + c];
                A[(size_t)r1 * n + c] = b;
                A[(size_t)r2 * n + c] = a;
            }
        }
    }
}

// U12 = L11^-1 A12 for one slab of TRSM_COLS columns per CTA.
constexpr int TRSM_COLS = 64;
constexpr int TRSM_THREADS = 256;
__global__ void __launch_bounds__(TRSM_THREADS, 1)
lu_trsm_kernel(double* __restrict__ A, int n, int k, int jb, int col_begin, int col_end) {
    extern __shared__ double smem[];
    double* L = smem;                              // [jb][PANEL_LD]
    double* S = smem + (size_t)LU_NB * PANEL_LD;   // [jb][TRSM_COLS]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = TRSM_THREADS / 32;
    const int c0 = col_begin + blockIdx.x * TRSM_COLS;
    const int nc = min(TRSM_COLS, col_end - c0);
    for (int idx = tid; idx < jb * jb; idx += TRSM_THREADS) {
        const int i = idx / jb, c = idx - i * jb;
        L[i * PANEL_LD + c] = A[(size_t)(k + i) * n + k + c];
    }
    for (int idx = tid; idx < jb * TRSM_COLS; idx += TRSM_THREADS) {
        const int i = idx / TRSM_COLS, c = idx - i * TRSM_COLS;
        S[i * TRSM_COLS + c] = c < nc ? A[(size_t)(k + i) * n + c0 + c] : 0.0;
    }
    __syncthreads();
    for (int t = 0; t + 1 < jb; ++t) {
        for (int i = t + 1 + warp; i < jb; i += nwarps) {
            const double l = L[i * PANEL_LD + t];
            S[i * TRSM_COLS + lane] = fma(-l, S[t * TRSM_COLS + lane], S[i * TRSM_COLS + lane]);
            S[i * TRSM_COLS + lane + 32] = fma(-l, S[t * TRSM_COLS + lane + 32], S[i * TRSM_COLS + lane + 32]);
        }
        __syncthreads();
    }
    for (int idx = tid; idx < jb * TRSM_COLS; idx += TRSM_THREADS) {
        const int i = idx / TRSM_COLS, c = idx - i * TRSM_COLS;
        if (c < nc) A[(size_t)(k + i) * n + c0 + c] = S[i * TRSM_COLS + c];
    }
}

// ---------------------------------------------------------------- DMMA trailing update
// C[M x N] -= Amat[M x K] * Bmat[K x N], all row-major with leading dimension ld.
constexpr int GM_BM = 128, GM_BK = 32;
constexpr int GM_THREADS = 256;
constexpr int GM_LDA = GM_BK + 4;    // 36: (row * 36 + col) hits 16 distinct 8-byte banks per half warp
template <int TN> struct GemmCfg {
    static constexpr int BN = 16 * TN;                 // 2 warps across N, TN 8-column groups each
    static constexpr int LDB = BN + 4;                 // same bank argument for the B fragments
    static constexpr int STAGE = GM_BM * GM_LDA + GM_BK * LDB;   // doubles per stage
    static constexpr int MINB = TN <= 4 ? 2 : 1;       // CTAs per SM the register budget allows
};

__device__ __forceinline__ void cp_async8(double* dst_smem, const double* src, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int bytes = pred ? 8 : 0;   // src-size 0 -> zero fill
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(src), "r"(bytes));
}
__device__ __forceinline__ void cp_async16(double* dst_smem, const double* src, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int bytes = pred ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(src), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma_8x8x4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// C[M x N] -= Amat[M x K] * Bmat[K x N], all row-major with leading dimension ld.
// 8 warps as 4 (M) x 2 (N); warp tile 32 x (8 TN).  TN = 4: 128 x 64 tile, 64 accumulator
// registers, 2 CTAs/SM (one CTA's barrier / cp.async wait overlaps the other's DMMA).
// VEC2: ld and all offsets even -> 16-byte cp.async.
template <int TN, bool VEC2>
__global__ void __launch_bounds__(GM_THREADS, GemmCfg<TN>::MINB)
lu_gemm_kernel(double* __restrict__ C, const double* __restrict__ Amat, const double* __restrict__ Bmat,
               int M, int N, int K, int ld) {
    using Cfg = GemmCfg<TN>;
    extern __shared__ double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 3, wn = warp >> 2;
    const int m0 = blockIdx.y * GM_BM, n0 = blockIdx.x * Cfg::BN;
    const int nchunks = (K + GM_BK - 1) / GM_BK;

    auto load_chunk = [&](int chunk, int stage) {
        double* sA = smem + (size_t)stage * Cfg::STAGE;
        double* sB = sA + GM_BM * GM_LDA;
        const int k0 = chunk * GM_BK;
        if (VEC2) {
            for (int idx = tid; idx < GM_BM * GM_BK / 2; idx += GM_THREADS) {
                const int r = idx >> 4, c = (idx & 15) * 2;
                const bool ok = (m0 + r < M) && (k0 + c < K);
                cp_async16(&sA[r * GM_LDA + c], ok ? &Amat[(size_t)(m0 + r) * ld + k0 + c] : Amat, ok);
            }
            for (int idx = tid; idx < GM_BK * Cfg::BN / 2; idx += GM_THREADS) {
                const int r = idx / (Cfg::BN / 2), c = (idx % (Cfg::BN / 2)) * 2;
                const bool ok = (k0 + r < K) && (n0 + c < N);
                cp_async16(&sB[r * Cfg::LDB + c], ok ? &Bmat[(size_t)(k0 + r) * ld + n0 + c] : Bmat, ok);
            }
        } else {
            for (int idx = tid; idx < GM_BM * GM_BK; idx += GM_THREADS) {
                const int r = idx >> 5, c = idx & 31;
                const bool ok = (m0 + r < M) && (k0 + c < K);
                cp_async8(&sA[r * GM_LDA + c], ok ? &Amat[(size_t)(m0 + r) * ld + k0 + c] : Amat, ok);
            }
            for (int idx = tid; idx < GM_BK * Cfg::BN; idx += GM_THREADS) {
                const int r = idx / Cfg::BN, c = idx % Cfg::BN;
                const bool ok = (k0 + r < K) && (n0 + c < N);
                cp_async8(&sB[r * Cfg::LDB + c], ok ? &Bmat[(size_t)(k0 + r) * ld + n0 + c] : Bmat, ok);
            }
        }
        cp_async_commit();
    };

    double acc[4][TN][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    load_chunk(0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
        if (ch + 1 < nchunks) {
            load_chunk(ch + 1, (ch + 1) & 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const double* sA = smem + (size_t)(ch & 1) * Cfg::STAGE;
        const double* sB = sA + GM_BM * GM_LDA;
#pragma unroll
        for (int kk = 0; kk < GM_BK; kk += 4) {
            double af[4], bf[TN];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                af[i] = sA[(wm * 32 + i * 8 + (lane >> 2)) * GM_LDA + kk + (lane & 3)];
#pragma unroll
            for (int j = 0; j < TN; ++j)
                bf[j] = sB[(kk + (lane & 3)) * Cfg::LDB + wn * (8 * TN) + j * 8 + (lane >> 2)];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) dmma_8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncthreads();
    }
    // epilogue: C -= acc
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = m0 + wm * 32 + i * 8 + (lane >> 2);
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int c = n0 + wn * (8 * TN) + j * 8 + (lane & 3) * 2;
            double* p = &C[(size_t)r * ld + c];
            if (VEC2) {
                if (c + 1 < N) {
                    double2 v = *reinterpret_cast<double2*>(p);
                    v.x -= acc[i][j][0]; v.y -= acc[i][j][1];
                    *reinterpret_cast<double2*>(p) = v;
                } else if (c < N) {
                    p[0] -= acc[i][j][0];
                }
            } else {
                if (c < N) p[0] -= acc[i][j][0];
                if (c + 1 < N) p[1] -= acc[i][j][1];
            }
        }
    }
}

template <int TN, bool VEC2>
static int launch_gemm(double* C, const double* A, const double* B, int M, int N, int K, int ld, cudaStream_t st) {
    using Cfg = GemmCfg<TN>;
    const size_t smem = sizeof(double) * 2 * (size_t)Cfg::STAGE;
    CUDA_TRY(cudaFuncSetAttribute(lu_gemm_kernel<TN, VEC2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((N + Cfg::BN - 1) / Cfg::BN, (M + GM_BM - 1) / GM_BM);
    lu_gemm_kernel<TN, VEC2><<<grid, GM_THREADS, smem, st>>>(C, A, B, M, N, K, ld);
    KERNEL_CHECK();
    return NODAL_OK;
}

// ---------------------------------------------------------------- solve phase
__global__ void __launch_bounds__(256, 1)
lu_apply_pivots_kernel(const double* __restrict__ b, double* __restrict__ x, const int* __restrict__ ipiv,
                       int n, int use_smem) {
    extern __shared__ double sx[];
    double* v = use_smem ? sx : x;
    for (int i = threadIdx.x; i < n; i += blockDim.x) v[i] = b[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < n; ++i) {
            const int p = ipiv[i];
            if (p != i) { const double t = v[i]; v[i] = v[p]; v[p] = t; }
        }
    }
    __syncthreads();
    if (use_smem)
        for (int i = threadIdx.x; i < n; i += blockDim.x) x[i] = v[i];
}

// Solves with the jb x jb diagonal block at (kb, kb): lower (unit) or upper.
__global__ void __launch_bounds__(LU_NB, 1)
lu_trsv_diag_kernel(const double* __restrict__ A, int n, int kb, int jb, double* __restrict__ x, int lower) {
    extern __shared__ double smem[];
    double* T = smem;                       // [jb][PANEL_LD]
    double* xs = smem + (size_t)LU_NB * PANEL_LD;
    const int tid = threadIdx.x;
    for (int idx = tid; idx < jb * jb; idx += LU_NB) {
        const int i = idx / jb, c = idx - i * jb;
        T[i * PANEL_LD + c] = A[(size_t)(kb + i) * n + kb + c];
    }
    if (tid < jb) xs[tid] = x[kb + tid];
    __syncthreads();
    if (lower) {
        for (int t = 0; t + 1 < jb; ++t) {
            if (tid > t && tid < jb) xs[tid] = fma(-T[tid * PANEL_LD + t], xs[t], xs[tid]);
            __syncthreads();
        }
    } else {
        for (int t = jb - 1; t >= 0; --t) {
            if (tid == t) xs[t] = xs[t] / T[t * PANEL_LD + t];
            __syncthreads();
            if (tid < t) xs[tid] = fma(-T[tid * PANEL_LD + t], xs[t], xs[tid]);
            __syncthreads();
        }
    }
    if (tid < jb) x[kb + tid] = xs[tid];
}

// x[r] -= A[r, cb : cb+jb] . x[cb : cb+jb] for r in [rb, re): one warp per row.
__global__ void __launch_bounds__(256)
lu_gemv_sub_kernel(const double* __restrict__ A, int n, int rb, int re, int cb, int jb,
                   double* __restrict__ x) {
    __shared__ double xs[LU_NB];
    for (int i = threadIdx.x; i < jb; i += blockDim.x) xs[i] = x[cb + i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int r = rb + warp; r < re; r += nwarps) {
        double s = 0.0;
        for (int c = lane; c < jb; c += 32) s = fma(A[(size_t)r * n + cb + c], xs[c], s);
        s = warp_sum(s);
        if (lane == 0) x[r] -= s;
    }
}

// Workspace nodal_lu_factor needs in the context arena besides the pivot vector.
static size_t lu_factor_scratch_bytes(int sms) {
    return sizeof(int) * 64 + sizeof(PivotCand) * 2 * (size_t)sms + sizeof(double) * (2 * (size_t)sms * LU_NB + 2 * LU_NB) +
           8192;
}

static int lu_check_size(nodal_ctx* ctx, int n, const char* what) {
    const int max_rows_per_cta = (226 * 1024 - 4096) / (PANEL_LD * 8) - 1;   // shared-memory limit
    if ((int64_t)n > (int64_t)ctx->num_sms * max_rows_per_cta) {
        nodal_set_error("%s: n=%d exceeds the panel capacity of this build (%d)", what, n,
                        ctx->num_sms * max_rows_per_cta);
        return NODAL_BAD_ARG;
    }
    return NODAL_OK;
}

// Factors G in place (P G = L U) on `st`; the scratch is carved from the arena, which the caller has
// reserved.  Returns NODAL_SINGULAR with *info_h set on an exactly zero pivot.
static int lu_factor_core(nodal_ctx* ctx, int n, double* G, int* ipiv, int32_t* info_h, cudaStream_t st) {
    const int sms = ctx->num_sms;
    int* info = carve<int>(ctx, 16);
    PivotCand* cand = carve<PivotCand>(ctx, 2 * (size_t)sms);
    double* candrow = carve<double>(ctx, 2 * (size_t)sms * LU_NB);
    double* diagrow = carve<double>(ctx, 2 * LU_NB);
    if (!ipiv || !info || !cand || !candrow || !diagrow) return NODAL_CUDA_ERROR;
    CUDA_TRY(cudaMemsetAsync(info, 0, sizeof(int), st));

    const size_t trsm_smem = sizeof(double) * ((size_t)LU_NB * PANEL_LD + (size_t)LU_NB * TRSM_COLS);
    {
        CUDA_TRY(cudaFuncSetAttribute(lu_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        CUDA_TRY(cudaFuncSetAttribute(lu_trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trsm_smem));
    }

    // Right-looking LU: after panel k, the row interchanges left of it, the update of the columns
    // right of it, then panel k+1.  One panel of look-ahead (panel k+1 on a second, high-priority
    // stream while the rest of step k runs) was measured on B200 (round 2) and removed: no gain,
    // 261 vs 252 ms at n = 16 384 -- the cooperative panel grid (one CTA per SM, ~117 KB of shared
    // memory each) does not become co-resident next to the DMMA update's two 108 KB CTAs per SM, so
    // the two kernels still ran back to back and the split update only added launches.
    auto launch_panel = [&](int k) -> int {
        int jb = std::min(LU_NB, n - k);
        int m = n - k;
        int rows_per_cta = std::max(32, (m + sms - 1) / sms);
        int ncta = (m + rows_per_cta - 1) / rows_per_cta;
        size_t panel_smem = sizeof(double) * ((size_t)rows_per_cta * PANEL_LD + LU_NB);
        double* Aptr = G;
        int n_ = n, k_ = k;
        void* args[] = {&Aptr, &n_, &k_, &jb, &rows_per_cta, &ipiv, &cand, &candrow, &diagrow, &info};
        CUDA_TRY(cudaLaunchCooperativeKernel((void*)lu_panel_kernel, dim3(ncta), dim3(PANEL_THREADS), args,
                                             panel_smem, st));
        ++g_nodal_launches;
        return NODAL_OK;
    };
    // step k applied to the columns [c0, c1): row interchanges, U12 = L11^-1 A12, A22 -= L21 U12
    auto update_cols = [&](int k, int jb, int c0, int c1, bool right_of_panel) -> int {
        if (c1 <= c0) return NODAL_OK;
        const int grid = std::min((c1 - c0 + 255) / 256, sms * 4);
        lu_swap_rows_kernel<<<grid, 256, 0, st>>>(G, n, k, jb, ipiv, c0, c1);
        KERNEL_CHECK();
        if (!right_of_panel) return NODAL_OK;
        const int rest = n - k - jb;
        lu_trsm_kernel<<<(c1 - c0 + TRSM_COLS - 1) / TRSM_COLS, TRSM_THREADS, trsm_smem, st>>>(G, n, k, jb, c0, c1);
        KERNEL_CHECK();
        double* Cp = G + (size_t)(k + jb) * n + c0;
        const double* Ap = G + (size_t)(k + jb) * n + k;
        const double* Bp = G + (size_t)k * n + c0;
        // all offsets are even when n is even (k, jb, c0 are multiples of 2): 16-byte copies
        const bool vec2 = (n % 2 == 0) && (((uintptr_t)G & 15) == 0) && (jb % 2 == 0) && (c0 % 2 == 0);
        if (vec2) NODAL_TRY((launch_gemm<4, true>(Cp, Ap, Bp, rest, c1 - c0, jb, n, st)));
        else NODAL_TRY((launch_gemm<4, false>(Cp, Ap, Bp, rest, c1 - c0, jb, n, st)));
        return NODAL_OK;
    };
    NODAL_TRY(launch_panel(0));
    for (int k = 0; k < n; k += LU_NB) {
        const int jb = std::min(LU_NB, n - k);
        const int right = k + jb;                       // first column right of the panel
        NODAL_TRY(update_cols(k, jb, 0, k, false));
        if (right >= n) break;
        NODAL_TRY(update_cols(k, jb, right, n, true));
        NODAL_TRY(launch_panel(right));
    }
    int* info_pinned = reinterpret_cast<int*>(ctx->pinned);
    CUDA_TRY(cudaMemcpyAsync(info_pinned, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (*info_pinned != 0) {
        *info_h = *info_pinned;
        return NODAL_SINGULAR;
    }
    return NODAL_OK;
}

// x = U^-1 L^-1 P rhs with the factors of lu_factor_core; enqueued on `st`.
static int lu_solve_core(nodal_ctx* ctx, int n, const double* G, const int* ipiv, const double* rhs, double* x,
                         cudaStream_t st) {
    const int sms = ctx->num_sms;
    const size_t trsv_smem = sizeof(double) * ((size_t)LU_NB * PANEL_LD + LU_NB);
    CUDA_TRY(cudaFuncSetAttribute(lu_trsv_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trsv_smem));
    CUDA_TRY(cudaFuncSetAttribute(lu_apply_pivots_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    const int use_smem = (size_t)n * 8 <= 200 * 1024;
    lu_apply_pivots_kernel<<<1, 256, use_smem ? (size_t)n * 8 : 0, st>>>(rhs, x, ipiv, n, use_smem);
    KERNEL_CHECK();
    for (int kb = 0; kb < n; kb += LU_NB) {
        const int jb = std::min(LU_NB, n - kb);
        lu_trsv_diag_kernel<<<1, LU_NB, trsv_smem, st>>>(G, n, kb, jb, x, 1);
        KERNEL_CHECK();
        const int rb = kb + jb;
        if (rb < n) {
            lu_gemv_sub_kernel<<<std::min((n - rb + 7) / 8, sms * 8), 256, 0, st>>>(G, n, rb, n, kb, jb, x);
            KERNEL_CHECK();
        }
    }
    for (int kb = ((n - 1) / LU_NB) * LU_NB; kb >= 0; kb -= LU_NB) {
        const int jb = std::min(LU_NB, n - kb);
        lu_trsv_diag_kernel<<<1, LU_NB, trsv_smem, st>>>(G, n, kb, jb, x, 0);
        KERNEL_CHECK();
        if (kb > 0) {
            lu_gemv_sub_kernel<<<std::min((kb + 7) / 8, sms * 8), 256, 0, st>>>(G, n, 0, kb, kb, jb, x);
            KERNEL_CHECK();
        }
    }
    return NODAL_OK;
}

extern "C" int nodal_lu_solve(nodal_ctx* ctx, int32_t n, double* G, const double* rhs, double* x,
                              int32_t* info_h, void* stream) {
    NvtxRange nvtx_range("nodal_lu_solve");
    if (!ctx || n < 0 || !info_h) return NODAL_BAD_ARG;
    *info_h = 0;
    if (n == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    NODAL_TRY(lu_check_size(ctx, n, "nodal_lu_solve"));
    NODAL_TRY(ctx_reserve(ctx, sizeof(int) * (size_t)n + lu_factor_scratch_bytes(ctx->num_sms)));
    int* ipiv = carve<int>(ctx, (size_t)n);
    NODAL_TRY(lu_factor_core(ctx, n, G, ipiv, info_h, st));
    NODAL_TRY(lu_solve_core(ctx, n, G, ipiv, rhs, x, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return NODAL_OK;
}

extern "C" int nodal_lu_factor(nodal_ctx* ctx, int32_t n, double* G, int32_t* ipiv, int32_t* info_h, void* stream) {
    NvtxRange nvtx_range("nodal_lu_factor");
    if (!ctx || n < 0 || !info_h || (n > 0 && (!G || !ipiv))) return NODAL_BAD_ARG;
    *info_h = 0;
    if (n == 0) return NODAL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    NODAL_TRY(lu_check_size(ctx, n, "nodal_lu_factor"));
    NODAL_TRY(ctx_reserve(ctx, lu_factor_scratch_bytes(ctx->num_sms)));
    return lu_factor_core(ctx, n, G, ipiv, info_h, st);
}

extern "C" int nodal_lu_solve_factored(nodal_ctx* ctx, int32_t n, const double* LU, const int32_t* ipiv,
                                       const double* rhs, double* x, void* stream) {
    NvtxRange nvtx_range("nodal_lu_solve_factored");
    if (!ctx || n < 0 || (n > 0 && (!LU || !ipiv || !rhs || !x))) return NODAL_BAD_ARG;
    if (n == 0) return NODAL_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    return lu_solve_core(ctx, n, LU, ipiv, rhs, x, (cudaStream_t)stream);
}

// Measurement aid (SURVEY.md section 8(d): "measure an FP64 GEMM-shaped peak on the box"): the
// trailing-update kernel of the LU on its own, C[M x N] -= A[M x K] B[K x N] (row-major, leading
// dimension ld, even), `reps` launches between two CUDA events on `stream`.  K = 128 is the shape
// the LU uses (one panel); a large K shows what the DMMA pipe sustains when the C tile is
// re-used, i.e. the denominator for the dense path's roofline.
extern "C" int nodal_dgemm_sub_profile(nodal_ctx* ctx, double* Cm, const double* Am, const double* Bm, int32_t M,
                                       int32_t N, int32_t K, int32_t ld, int32_t reps, double* ms_out, void* stream) {
    if (!ctx || !Cm || !Am || !Bm || !ms_out || M < 1 || N < 1 || K < 1 || reps < 1 || (ld & 1)) return NODAL_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    int rc = NODAL_OK;
    for (int k = -2; k < reps && rc == NODAL_OK; ++k) {
        if (k == 0) cudaEventRecord(e0, st);
        rc = launch_gemm<4, true>(Cm, Am, Bm, M, N, K, ld, st);
    }
    cudaEventRecord(e1, st);
    float ms = 0.f;
    if (cudaEventSynchronize(e1) == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
    *ms_out = ms / reps;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return rc;
}
