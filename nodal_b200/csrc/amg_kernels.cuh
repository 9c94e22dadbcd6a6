// Device kernels of the aggregation AMG (setup + V-cycle + CG vector updates), shared by the
// single-GPU driver (amg.cu) and the row-partitioned multi-GPU driver (dist_amg.cu).
// See amg.cu for the algorithm notes.
#pragma once
#include "amg_core.cuh"
#include "amg_merge_core.cuh"
#include "sparse.cuh"

constexpr int AT = 256;

// ------------------------------------------------------------------ setup kernels
#define ROW_LOOP(i, n)                                                              \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)(n); \
         i += (int64_t)gridDim.x * blockDim.x)

static __global__ void __launch_bounds__(AT)
amg_propose_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                   const double* __restrict__ data, const int32_t* __restrict__ match,
                   int32_t* __restrict__ best, int32_t nown, int32_t base) {
    ROW_LOOP(i, n) best[i] = match[i] >= 0 ? -1 : amg_pick((int32_t)i, indptr, indices, data, match, nown, base);
}

static __global__ void __launch_bounds__(AT)
amg_accept_kernel(int32_t n, const int32_t* __restrict__ best, int32_t* __restrict__ match) {
    ROW_LOOP(i, n) {
        if (match[i] >= 0) continue;
        const int32_t b = best[i];
        if (b >= 0 && best[b] == (int32_t)i) match[i] = b;
    }
}

static __global__ void __launch_bounds__(AT)
amg_root_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                const double* __restrict__ data, const int32_t* __restrict__ match,
                int32_t* __restrict__ root, u32* __restrict__ leader, int32_t nown, int32_t base) {
    ROW_LOOP(i, n) {
        const int32_t r = amg_root((int32_t)i, indptr, indices, data, match, nown, base);
        root[i] = r;
        leader[i] = r == (int32_t)i ? 1u : 0u;
    }
}

static __global__ void __launch_bounds__(AT)
amg_assign_kernel(int32_t n, const int32_t* __restrict__ root, const u32* __restrict__ ids,
                  int32_t* __restrict__ agg) {
    ROW_LOOP(i, n) agg[i] = (int32_t)ids[root[i]];
}

static __global__ void __launch_bounds__(AT)
amg_compose_kernel(int32_t n, int32_t* __restrict__ comp, const int32_t* __restrict__ next) {
    ROW_LOOP(i, n) comp[i] = next[comp[i]];
}

static __global__ void __launch_bounds__(AT)
amg_relabel_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                   const double* __restrict__ data, const int32_t* __restrict__ agg, int cb,
                   u64* __restrict__ keys, double* __restrict__ vals) {
    ROW_LOOP(i, n) {
        const u64 hi = (u64)agg[i] << cb;
        const int32_t e = indptr[i + 1];
        for (int32_t p = indptr[i]; p < e; ++p) {
            keys[p] = hi | (u64)agg[indices[p]];
            vals[p] = data[p];
        }
    }
}

static __global__ void __launch_bounds__(AT)
amg_pt_keys_kernel(int32_t n, const int32_t* __restrict__ agg, int cb, u64* __restrict__ keys,
                   double* __restrict__ vals) {
    ROW_LOOP(i, n) {
        keys[i] = ((u64)agg[i] << cb) | (u64)i;
        vals[i] = 1.0;
    }
}

// ------------------------------------------------------------------ coarsest level: explicit inverse
// [A | I] -> [I | A^-1] by Gauss-Jordan without pivoting (A is symmetric positive definite),
// one launch per pivot, ping-pong between two n x 2n buffers so a step has no read/write race.
static __global__ void __launch_bounds__(AT)
amg_dense_init_kernel(int32_t n, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                      const double* __restrict__ data, double* __restrict__ M) {
    const int64_t W = 2 * (int64_t)n;
    ROW_LOOP(i, n) {
        M[i * W + n + i] = 1.0;
        const int32_t e = indptr[i + 1];
        for (int32_t p = indptr[i]; p < e; ++p) M[i * W + indices[p]] = data[p];
    }
}

static __global__ void __launch_bounds__(AT)
amg_gj_step_kernel(int32_t n, int32_t k, const double* __restrict__ src, double* __restrict__ dst,
                   int* __restrict__ bad) {
    const int64_t W = 2 * (int64_t)n;
    const double piv = src[k * W + k];
    if (blockIdx.x == 0 && threadIdx.x == 0 && !(piv > 0.0) && *bad == 0) *bad = k + 1;
    ROW_LOOP(idx, (int64_t)n * W) {
        const int64_t i = idx / W, j = idx - i * W;
        const double rkj = src[k * W + j] / piv;
        dst[idx] = i == k ? rkj : src[idx] - src[i * W + k] * rkj;
    }
}

static __global__ void __launch_bounds__(AT)
amg_dense_extract_kernel(int32_t n, const double* __restrict__ M, double* __restrict__ inv) {
    const int64_t W = 2 * (int64_t)n;
    ROW_LOOP(idx, (int64_t)n * n) {
        const int64_t i = idx / n, j = idx - i * n;
        inv[idx] = M[i * W + n + j];
    }
}

// x = inv b, one warp per row
static __global__ void __launch_bounds__(AT)
amg_gemv_kernel(int32_t n, const double* __restrict__ inv, const double* __restrict__ b,
                double* __restrict__ x) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += nwarps) {
        double acc = 0.0;
        for (int32_t j = lane; j < n; j += 32) acc = fma(inv[r * n + j], b[j], acc);
        acc = warp_sum(acc);
        if (lane == 0) x[r] = acc;
    }
}

// ------------------------------------------------------------------ cycle kernels
static __global__ void __launch_bounds__(AT)
amg_jacobi0_kernel(int32_t n, const double* __restrict__ dinv, const double* __restrict__ b,
                   double omega, double* __restrict__ x) {
    ROW_LOOP(i, n) x[i] = amg_jacobi_start(omega, dinv[i], b[i]);
}

// SELL-32 sweep, one warp per slice.
//   MODE 0: y = A x, per-block partial sums of x.y        (CG: q = A p, p.q)
//   MODE 1: y = b - A x                                   (residual)
//   MODE 2: y = x + omega D^-1 (b - A x)                  (damped Jacobi sweep, out of place)
template <int MODE, class A>
static __global__ void __launch_bounds__(AT, 5)
amg_sell_kernel(int32_t n, int32_t nslices, const u32* __restrict__ slice_w, A a0,
                const double* __restrict__ dinv, const double* __restrict__ b,
                const double* __restrict__ x, double omega, double* __restrict__ y,
                double* __restrict__ part) {
    const A a = a0.staged();
    __shared__ double red[33];
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double dot = 0.0;
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int w = (int)(slice_w[s + 1] - w0);
        const int64_t r = s * 32 + lane;
        const double acc = sell_row_dot(a, (int64_t)w0 * 32 + lane, r, w, x);
        if (r < n) {
            if (MODE == 0) { y[r] = acc; dot = fma(x[r], acc, dot); }
            if (MODE == 1) y[r] = amg_residual(b[r], acc);
            if (MODE == 2) y[r] = amg_jacobi_update(omega, dinv[r], b[r], acc, x[r]);
        }
    }
    if (MODE == 0) {
        const double t = block_sum(dot, red);
        if (threadIdx.x == 0) part[blockIdx.x] = t;
    }
}

// bc[I] = sum of r over the members of aggregate I, in increasing row order
static __global__ void __launch_bounds__(AT)
amg_restrict_kernel(int32_t nc, const int32_t* __restrict__ pt_ptr, const int32_t* __restrict__ pt_idx,
                    const double* __restrict__ r, double* __restrict__ bc) {
    ROW_LOOP(I, nc) {
        double s = 0.0;
        const int32_t e = pt_ptr[I + 1];
        for (int32_t p = pt_ptr[I]; p < e; ++p) s += r[pt_idx[p]];
        bc[I] = s;
    }
}

static __global__ void __launch_bounds__(AT)
amg_prolong_kernel(int32_t n, const int32_t* __restrict__ agg, const double* __restrict__ xc,
                   double scale, const double* __restrict__ x, double* __restrict__ xa) {
    ROW_LOOP(i, n) xa[i] = amg_prolong_add(scale, xc[agg[i]], x[i]);
}

// The V-cycle's sweeps with the vector they multiply formed at every gathered column instead of
// stored by a kernel of its own (jacobi0 before MODE 1, prolong before MODE 2); same rounding steps
// (amg_cycle_core.cuh), so y is bit for bit what the unfused pair computes.
//   MODE 1: y = b - A x0                          x0 = omega D^-1 b      (residual of the Jacobi start)
//   MODE 2: y = x~ + omega D^-1 (b - A x~)        x~ = x0 + scale P xc   (post-smoothing)
struct JacobiStartAt {
    const double* __restrict__ dinv;
    const double* __restrict__ b;
    double omega;
    __device__ __forceinline__ double operator()(int32_t c) const {
        return amg_jacobi_start(omega, __ldg(&dinv[c]), __ldg(&b[c]));
    }
};

struct ProlongatedAt {
    JacobiStartAt x0;
    const int32_t* __restrict__ agg;
    const double* __restrict__ xc;
    double scale;
    __device__ __forceinline__ double operator()(int32_t c) const {
        return amg_prolong_add(scale, __ldg(&xc[__ldg(&agg[c])]), x0(c));
    }
};

template <int MODE, class A>
static __global__ void __launch_bounds__(AT, 5)
amg_cycle_sweep_kernel(int32_t n, int32_t nslices, const u32* __restrict__ slice_w, A a0,
                       const double* __restrict__ dinv, const double* __restrict__ b, double omega,
                       const int32_t* __restrict__ agg, const double* __restrict__ xc, double scale,
                       double* __restrict__ y) {
    const A a = a0.staged();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const JacobiStartAt x0{dinv, b, omega};
    const ProlongatedAt xa{x0, agg, xc, scale};
    for (int64_t s = warp; s < nslices; s += nwarps) {
        const u32 w0 = slice_w[s];
        const int w = (int)(slice_w[s + 1] - w0);
        const int64_t base = (int64_t)w0 * 32 + lane;
        const int64_t r = s * 32 + lane;
        if (MODE == 1) {
            const double acc = sell_row_gather(a, base, r, w, x0);
            if (r < n) y[r] = amg_residual(b[r], acc);
        }
        if (MODE == 2) {
            const double acc = sell_row_gather(a, base, r, w, xa);
            if (r < n) y[r] = amg_jacobi_update(omega, dinv[r], b[r], acc, xa((int32_t)r));
        }
    }
}

// ------------------------------------------------------------------ CG vector kernels
static __global__ void __launch_bounds__(AT)
apcg_dot_kernel(int32_t n, const double* __restrict__ a, const double* __restrict__ b,
                double* __restrict__ part) {
    __shared__ double red[33];
    double t = 0.0;
    ROW_LOOP(i, n) t = fma(a[i], b[i], t);
    t = block_sum(t, red);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
}

static __global__ void __launch_bounds__(AT)
apcg_sum_kernel(const double* __restrict__ part, int count, double* __restrict__ out) {
    __shared__ double red[33];
    const double t = reduce_partials(part, count, red);
    if (threadIdx.x == 0) out[0] = t;
}

// alpha = rz / p.q ; x += alpha p ; r -= alpha q ; partial sums of r.r
static __global__ void __launch_bounds__(AT)
apcg_update_kernel(int32_t n, const double* __restrict__ part_pq, int npq, const double* __restrict__ rz,
                   const double* __restrict__ p, const double* __restrict__ q, double* __restrict__ x,
                   double* __restrict__ r, double* __restrict__ part_rr) {
    __shared__ double red[33];
    const double pq = reduce_partials(part_pq, npq, red);
    const double alpha = rz[0] / pq;
    double t = 0.0;
    ROW_LOOP(i, n) {
        x[i] = fma(alpha, p[i], x[i]);
        const double ri = fma(-alpha, q[i], r[i]);
        r[i] = ri;
        t = fma(ri, ri, t);
    }
    t = block_sum(t, red);
    if (threadIdx.x == 0) part_rr[blockIdx.x] = t;
}

// rz' = r.z (from partials) ; beta = rz'/rz ; p = z + beta p
static __global__ void __launch_bounds__(AT)
apcg_direction_kernel(int32_t n, const double* __restrict__ part_rz, int nrz,
                      const double* __restrict__ rz_old, double* __restrict__ rz_new,
                      const double* __restrict__ z, double* __restrict__ p, int first) {
    __shared__ double red[33];
    const double rzn = reduce_partials(part_rz, nrz, red);
    const double beta = first ? 0.0 : rzn / rz_old[0];
    ROW_LOOP(i, n) p[i] = first ? z[i] : fma(beta, p[i], z[i]);
    if (blockIdx.x == 0 && threadIdx.x == 0) rz_new[0] = rzn;
}


// ------------------------------------------------------------------ sort-free setup kernels
// Members of every aggregate: count, scan, place (arrival order), then every aggregate sorts its
// own few members -- the result (rows in increasing order) does not depend on the atomics' order.
static __global__ void __launch_bounds__(AT)
amg_count_members_kernel(int32_t n, const int32_t* __restrict__ agg, u32* __restrict__ cnt) {
    ROW_LOOP(i, n) atomicAdd(&cnt[agg[i]], 1u);
}

static __global__ void __launch_bounds__(AT)
amg_place_members_kernel(int32_t n, const int32_t* __restrict__ agg, const int32_t* __restrict__ pt_ptr,
                         u32* __restrict__ cursor, int32_t* __restrict__ pt_idx) {
    ROW_LOOP(i, n) {
        const int32_t a = agg[i];
        pt_idx[pt_ptr[a] + (int32_t)atomicAdd(&cursor[a], 1u)] = (int32_t)i;
    }
}

static __global__ void __launch_bounds__(AT)
amg_sort_members_kernel(int32_t nc, const int32_t* __restrict__ pt_ptr, int32_t* __restrict__ pt_idx) {
    ROW_LOOP(I, nc) {
        const int32_t b = pt_ptr[I], e = pt_ptr[I + 1];
        for (int32_t p = b + 1; p < e; ++p) {
            const int32_t v = pt_idx[p];
            int32_t q = p;
            while (q > b && pt_idx[q - 1] > v) { pt_idx[q] = pt_idx[q - 1]; --q; }
            pt_idx[q] = v;
        }
    }
}

// Galerkin product by merging (amg_merge_core.cuh): upper bounds, rows into their slices, compaction.
static __global__ void __launch_bounds__(AT)
amg_merge_bound_kernel(int32_t nc, const int32_t* __restrict__ pt_ptr, const int32_t* __restrict__ pt_idx,
                       const int32_t* __restrict__ indptr, u32* __restrict__ bound) {
    ROW_LOOP(I, nc) bound[I] = (u32)amg_merge_bound((int32_t)I, pt_ptr, pt_idx, indptr);
}

static __global__ void __launch_bounds__(AT)
amg_merge_rows_kernel(int32_t nc, const int32_t* __restrict__ pt_ptr, const int32_t* __restrict__ pt_idx,
                      const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                      const double* __restrict__ data, const int32_t* __restrict__ label, int32_t ncol_limit,
                      const u32* __restrict__ off, int32_t* tmp_cols, double* tmp_vals, u32* __restrict__ kept) {
    // Short rows (the common case: 2 - 3 member rows of 5 - 9 entries) are merged in a thread-local
    // list and written out once; the insertion's read-backs otherwise go to the global slice.
    constexpr int LOCAL = 32;
    ROW_LOOP(I, nc) {
        const u32 o = off[I];
        if (off[I + 1] - o <= (u32)LOCAL) {
            int32_t lc[LOCAL];
            double lv[LOCAL];
            const int32_t k = amg_merge_row((int32_t)I, pt_ptr, pt_idx, indptr, indices, data, label, lc, lv, ncol_limit);
            for (int32_t e = 0; e < k; ++e) { tmp_cols[o + e] = lc[e]; tmp_vals[o + e] = lv[e]; }
            kept[I] = (u32)k;
        } else {
            kept[I] = (u32)amg_merge_row((int32_t)I, pt_ptr, pt_idx, indptr, indices, data, label, tmp_cols + o,
                                         tmp_vals + o, ncol_limit);
        }
    }
}

static __global__ void __launch_bounds__(AT)
amg_merge_compact_kernel(int32_t nc, const u32* __restrict__ off, const int32_t* __restrict__ out_ptr,
                         const int32_t* __restrict__ tmp_cols, const double* __restrict__ tmp_vals,
                         int32_t* __restrict__ out_cols, double* __restrict__ out_vals) {
    ROW_LOOP(I, nc) {
        const int32_t b = out_ptr[I], cnt = out_ptr[I + 1] - b;
        const u32 src = off[I];
        for (int32_t k = 0; k < cnt; ++k) {
            out_cols[b + k] = tmp_cols[src + k];
            out_vals[b + k] = tmp_vals[src + k];
        }
    }
}
