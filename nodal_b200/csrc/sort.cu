// Device-wide exclusive scan (u32) and stable LSD radix sort of (u64 key, u64 payload)
// pairs, hand written for the CSR build (no CUB / Thrust).
//
// Radix sort: 8-bit digits, one pass per digit over only the key bits in use.
//   1. onesweep_hist_kernel   digit histograms of all passes from one read of the keys
//   2. onesweep_bases_kernel  exclusive scan of each pass's histogram = first output slot of
//                             every digit
//   3. onesweep_pass_kernel   one kernel per pass: ranks the keys of a tile stably (warp
//                             match-any multi-split, warps own consecutive key ranges), finds
//                             the tile's output offsets by decoupled look-back, reorders the
//                             tile by digit in shared memory and writes every digit run to its
//                             place with coalesced stores.
// Stability: inside a tile, warp w owns keys [w*32*IPT, (w+1)*32*IPT) and visits them in
// rounds of 32 consecutive keys, so (warp, round, lane) order == input order.
#include <algorithm>

#include "common.cuh"

// ------------------------------------------------------------------ scan
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_IPT = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_IPT;

// exclusive scan of one value per thread across the block; returns exclusive prefix,
// *total = block total (valid in all threads).  smem: >= 34 u32.
__device__ __forceinline__ u32 block_excl_scan_u32(u32 v, u32* smem, u32* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    u32 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) smem[w] = inc;
    __syncthreads();
    if (w == 0) {
        u32 s = (lane < nw) ? smem[lane] : 0u;
        u32 si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= o) si += t;
        }
        if (lane < nw) smem[lane] = si - s;  // exclusive warp offsets
        if (lane == 31) smem[33] = si;       // block total (nw <= 32)
    }
    __syncthreads();
    const u32 res = smem[w] + inc - v;
    *total = smem[33];
    return res;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_tile_sums_kernel(const u32* __restrict__ in, int64_t count, u32* __restrict__ tile_sums) {
    __shared__ u32 sm[40];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_IPT; ++k) {
        const int64_t i = base + (int64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < count) s += in[i];
    }
    u32 total;
    block_excl_scan_u32(s, sm, &total);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// Scans one tile; adds tile_offsets[blockIdx.x] (may be null for a single tile).
__global__ void __launch_bounds__(SCAN_THREADS)
scan_tile_apply_kernel(const u32* __restrict__ in, u32* __restrict__ out, int64_t count,
                       const u32* __restrict__ tile_offsets, u32* __restrict__ total_out) {
    __shared__ u32 sm[40];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_IPT;
    u32 v[SCAN_IPT];
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_IPT; ++k) {
        const int64_t i = base + k;
        v[k] = (i < count) ? in[i] : 0u;
        s += v[k];
    }
    u32 total;
    u32 run = block_excl_scan_u32(s, sm, &total);
    const u32 off = tile_offsets ? tile_offsets[blockIdx.x] : 0u;
    run += off;
#pragma unroll
    for (int k = 0; k < SCAN_IPT; ++k) {
        const int64_t i = base + k;
        if (i < count) out[i] = run;
        run += v[k];
    }
    if (total_out && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *total_out = off + total;
}

static int64_t scan_tiles(int64_t count) { return (count + SCAN_TILE - 1) / SCAN_TILE; }

size_t scan_scratch_bytes(int64_t count) {
    size_t bytes = 0;
    int64_t c = count;
    while (c > SCAN_TILE) {
        c = scan_tiles(c);
        bytes += align_up((size_t)c * sizeof(u32), 256) + 256;
    }
    return bytes + 512;
}

// in and out may alias.  total_dev (optional) receives the grand total.
int scan_exclusive_u32(nodal_ctx* ctx, const u32* in, u32* out, int64_t count, u32* total_dev,
                       cudaStream_t st) {
    if (count <= 0) {
        if (total_dev) CUDA_TRY(cudaMemsetAsync(total_dev, 0, sizeof(u32), st));
        return NODAL_OK;
    }
    const int64_t tiles = scan_tiles(count);
    if (tiles == 1) {
        scan_tile_apply_kernel<<<1, SCAN_THREADS, 0, st>>>(in, out, count, nullptr, total_dev);
        KERNEL_CHECK();
        return NODAL_OK;
    }
    u32* sums = carve<u32>(ctx, (size_t)tiles);
    if (!sums) return NODAL_CUDA_ERROR;
    scan_tile_sums_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, count, sums);
    KERNEL_CHECK();
    NODAL_TRY(scan_exclusive_u32(ctx, sums, sums, tiles, nullptr, st));
    scan_tile_apply_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, out, count, sums, total_dev);
    KERNEL_CHECK();
    return NODAL_OK;
}

// ------------------------------------------------------------------ radix sort
constexpr int RS_THREADS = 256;
constexpr int RS_BINS = 256;

// ------------------------------------------------------------------ single-pass-per-digit sort
// ("onesweep" class).  One upfront kernel builds the digit histograms of ALL passes from one read
// of the keys; every pass is then ONE kernel that reads keys + payload once, finds each tile's
// output offsets by decoupled look-back over per-tile digit counts (no global scan, no second
// read), reorders the tile by digit in shared memory -- keys and payload staged together -- and
// writes every digit run to its final place.  Stability: inside a tile (warp, round, lane) order
// is input order, tiles are ordered by the look-back.
// Tile ids are handed out by an atomic ticket, so a tile's predecessors have always started and
// the look-back cannot dead-lock; its spin is bounded anyway (error flag instead of a hang).
constexpr int OS_MAXPASS = 8;
constexpr u32 OS_AGG = 1u << 30, OS_INC = 2u << 30, OS_VAL = (1u << 30) - 1;
constexpr long long OS_SPIN_LIMIT = 4000000000ll;

__global__ void __launch_bounds__(RS_THREADS)
onesweep_hist_kernel(const u64* __restrict__ keys, int64_t count, int passes, u32* __restrict__ ghist) {
    __shared__ u32 h[OS_MAXPASS][RS_BINS];
    for (int i = threadIdx.x; i < OS_MAXPASS * RS_BINS; i += RS_THREADS) (&h[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t rounds = (count + stride - 1) / stride;            // warp-uniform trip count
    for (int64_t it = 0; it < rounds; ++it) {
        const int64_t i = it * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        const bool live = i < count;
        const u64 k = live ? keys[i] : 0ull;
        for (int p = 0; p < passes; ++p) {
            const u32 dg = (u32)(k >> (8 * p)) & 0xffu;
            // nearly sorted input puts a whole warp into one bin of the high digits: one add for all
            const u32 d0 = __shfl_sync(0xffffffffu, dg, 0);
            const bool same = __all_sync(0xffffffffu, live && dg == d0);
            if (same) { if (lane == 0) atomicAdd(&h[p][d0], 32u); }
            else if (live) atomicAdd(&h[p][dg], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < passes * RS_BINS; i += RS_THREADS) {
        const u32 v = (&h[0][0])[i];
        if (v) atomicAdd(&ghist[i], v);
    }
}

// ghist[p][*] -> exclusive scan in place (one block per pass)
__global__ void __launch_bounds__(RS_BINS)
onesweep_bases_kernel(u32* __restrict__ ghist) {
    __shared__ u32 sm[40];
    u32* row = ghist + (size_t)blockIdx.x * RS_BINS;
    u32 total;
    const u32 v = row[threadIdx.x];
    const u32 ex = block_excl_scan_u32(v, sm, &total);
    row[threadIdx.x] = ex;
}

// 512 threads x 8 keys per tile of 4096 at 2 CTAs / SM (32 resident warps).  History on the
// 16.8 M-row grid (134 M pairs, ncu, per pass): 256 x 16 keys at 128 registers, 2 CTAs / SM: 1.60 ms;
// 512 x 8 at 64 registers: 1.45 ms; + windowed look-back: 1.34 ms = 3.2 TB/s with DRAM traffic equal
// to the algorithmic 4.35 GB (round 1's three-kernel pass: 3.5 ms).  256 x 8 tiles at 4 CTAs / SM were
// slower again (1.47 ms): warps wait at the tile's barriers and on the loads in front of them in
// equal parts, so the next step is overlapping a tile's loads with the previous tile's scatter
// inside one CTA, not more CTAs.
constexpr int OS_THREADS = 512;
constexpr int OS_WARPS = OS_THREADS / 32;
constexpr int OS_IPT = 8;
constexpr int OS_TILE = OS_THREADS * OS_IPT;
constexpr int OS_LOOK = 8;
constexpr int OS_CTAS_PER_SM = 2;

__global__ void __launch_bounds__(OS_THREADS, OS_CTAS_PER_SM)
onesweep_pass_kernel(const u64* __restrict__ keys_in, const u64* __restrict__ vals_in,
                     u64* __restrict__ keys_out, u64* __restrict__ vals_out, int64_t count, int shift,
                     int64_t tiles, const u32* __restrict__ gbase /* [RS_BINS] exclusive */,
                     u32* desc /* [tiles][RS_BINS], zeroed */, u32* ticket /* zeroed */, int* err) {
    extern __shared__ u64 os_stage[];                 // [OS_TILE] keys | [OS_TILE] payload
    u64* stage_k = os_stage;
    u64* stage_v = os_stage + OS_TILE;
    __shared__ u32 warp_cnt[OS_WARPS][RS_BINS];      // per-warp digit counts -> exclusive offsets
    __shared__ u32 digit_start[RS_BINS];             // start of each digit run inside the tile
    __shared__ u32 digit_gbase[RS_BINS];             // global slot of the run's first element
    __shared__ u32 scan_sm[40];
    __shared__ int64_t s_tile;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u32 lt = lanemask_lt();

    for (;;) {
        __syncthreads();                             // previous tile's shared state is no longer read
        if (threadIdx.x == 0) s_tile = (int64_t)atomicAdd(ticket, 1u);
        for (int i = threadIdx.x; i < OS_WARPS * RS_BINS; i += OS_THREADS) (&warp_cnt[0][0])[i] = 0;
        __syncthreads();
        const int64_t tile = s_tile;
        if (tile >= tiles) break;
        const int64_t base = tile * OS_TILE + (int64_t)w * 32 * OS_IPT;

        u64 key[OS_IPT];
        u32 rank[OS_IPT];   // rank of the key among equal digits seen earlier by this warp
#pragma unroll
        for (int k = 0; k < OS_IPT; ++k) {
            const int64_t i = base + k * 32 + lane;
            key[k] = i < count ? keys_in[i] : 0ull;
        }
#pragma unroll
        for (int k = 0; k < OS_IPT; ++k) {
            const int64_t i = base + k * 32 + lane;
            const bool live = i < count;
            const u32 dg = live ? ((u32)(key[k] >> shift) & 0xffu) : 256u;
            const u32 peers = __match_any_sync(0xffffffffu, dg);
            const u32 before = live ? warp_cnt[w][dg] : 0u;
            __syncwarp();
            rank[k] = before + __popc(peers & lt);
            if (live && (peers & lt) == 0u) warp_cnt[w][dg] = before + __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        // per digit (threads 0 .. 255): exclusive prefix over warps, tile total, look-back
        const int dgt = threadIdx.x;
        u32 run = 0;
        volatile u32* mine = desc + (size_t)tile * RS_BINS + (dgt & (RS_BINS - 1));
        if (dgt < RS_BINS) {
#pragma unroll
            for (int ww = 0; ww < OS_WARPS; ++ww) {
                const u32 t = warp_cnt[ww][dgt];
                warp_cnt[ww][dgt] = run;
                run += t;
            }
            *mine = (tile == 0 ? OS_INC : OS_AGG) | run;
        }
        u32 total;
        const u32 start = block_excl_scan_u32(run, scan_sm, &total);
        if (dgt < RS_BINS) {
            digit_start[dgt] = start;
            u32 excl = 0;
            if (tile > 0) {
                // Look-back in windows of OS_LOOK predecessors whose descriptor loads are all in
                // flight at once: with ~300 tiles in flight the walk to the nearest inclusive
                // prefix is dozens of steps, and one dependent L2 round trip per step made the
                // look-back the longest phase of a tile.
                const long long t0 = clock64();
                bool done = false;
                for (int64_t t = tile - 1; t >= 0 && !done; t -= OS_LOOK) {
                    u32 v[OS_LOOK];
#pragma unroll
                    for (int k = 0; k < OS_LOOK; ++k) {
                        const int64_t tt = t - k;
                        v[k] = tt >= 0 ? *(const volatile u32*)(desc + (size_t)tt * RS_BINS + dgt) : OS_INC;
                    }
#pragma unroll
                    for (int k = 0; k < OS_LOOK; ++k) {
                        if (done) continue;
                        u32 x = v[k];
                        if ((x >> 30) == 0u) {
                            const volatile u32* p = desc + (size_t)(t - k) * RS_BINS + dgt;
                            x = *p;
                            while ((x >> 30) == 0u) {
                                if (clock64() - t0 > OS_SPIN_LIMIT) { *err = 1; x = OS_INC; break; }
                                x = *p;
                            }
                        }
                        excl += x & OS_VAL;
                        if ((x >> 30) == 2u) done = true;
                    }
                }
                *mine = OS_INC | (excl + run);
            }
            digit_gbase[dgt] = gbase[dgt] + excl;
        }
        __syncthreads();
        const int64_t tile_base = tile * OS_TILE;
        const int tile_n = (count - tile_base < OS_TILE) ? (int)(count - tile_base) : OS_TILE;
#pragma unroll
        for (int k = 0; k < OS_IPT; ++k) {
            const int64_t i = base + k * 32 + lane;
            if (i < count) {
                const u32 dg = (u32)(key[k] >> shift) & 0xffu;
                const u32 pos = digit_start[dg] + warp_cnt[w][dg] + rank[k];
                stage_k[pos] = key[k];
                stage_v[pos] = vals_in[i];
            }
        }
        __syncthreads();
        for (int j = threadIdx.x; j < tile_n; j += OS_THREADS) {
            const u64 kk = stage_k[j];
            const u32 dg = (u32)(kk >> shift) & 0xffu;
            const int64_t dst = (int64_t)digit_gbase[dg] + (j - (int)digit_start[dg]);
            keys_out[dst] = kk;
            vals_out[dst] = stage_v[j];
        }
    }
}

constexpr size_t RADIX_ERR_OFFSET = 3072;

int radix_sort_check(nodal_ctx* ctx) {
    int* err = reinterpret_cast<int*>(static_cast<char*>(ctx->pinned) + RADIX_ERR_OFFSET);
    if (*err) {
        *err = 0;
        nodal_set_error("radix sort: look-back timed out (device-side spin limit)");
        return NODAL_CUDA_ERROR;
    }
    return NODAL_OK;
}

size_t radix_sort_scratch_bytes(int64_t count) {
    const int64_t tiles = (count + OS_TILE - 1) / OS_TILE;
    const size_t desc = align_up(((size_t)tiles * RS_BINS + 64) * sizeof(u32), 256);
    return desc + align_up(OS_MAXPASS * RS_BINS * sizeof(u32), 256) + 1024;
}

// Sorts by key bits [0, bits).  Ping-pongs between (keys, vals) and (keys_alt, vals_alt);
// *result_in_alt tells where the sorted data ended up.
int radix_sort_pairs(nodal_ctx* ctx, u64* keys, u64* vals, u64* keys_alt, u64* vals_alt,
                     int64_t count, int bits, bool* result_in_alt, cudaStream_t st) {
    NvtxRange nvtx_range("radix_sort_pairs");
    *result_in_alt = false;
    if (count <= 1 || bits <= 0) return NODAL_OK;
    const int64_t tiles = (count + OS_TILE - 1) / OS_TILE;
    if (tiles * RS_BINS * 2 >= (int64_t)1 << 32 || count >= (int64_t)1 << 30) {
        nodal_set_error("radix_sort_pairs: too many elements");
        return NODAL_BAD_ARG;
    }
    const int passes = (bits + 7) / 8;
    if (passes > OS_MAXPASS) {
        nodal_set_error("radix_sort_pairs: keys wider than 64 bits");
        return NODAL_BAD_ARG;
    }
    u64 *src_k = keys, *src_v = vals, *dst_k = keys_alt, *dst_v = vals_alt;
    // tile descriptors + ticket + error word (zeroed before every pass), digit bases of all passes
    const size_t desc_words = (size_t)tiles * RS_BINS + 64;
    u32* desc = carve<u32>(ctx, desc_words);
    u32* ghist = carve<u32>(ctx, OS_MAXPASS * RS_BINS);
    if (!desc || !ghist) return NODAL_CUDA_ERROR;
    u32* ticket = desc + (size_t)tiles * RS_BINS;
    // look-back timeout flag: a word of the ctx's pinned host block (device-writable under UVA),
    // checked by radix_sort_check() after the caller's next stream synchronisation
    int* err = reinterpret_cast<int*>(static_cast<char*>(ctx->pinned) + RADIX_ERR_OFFSET);
    static bool attr_set = false;
    const size_t dyn = 2 * (size_t)OS_TILE * sizeof(u64);
    if (!attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(onesweep_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        attr_set = true;
    }
    CUDA_TRY(cudaMemsetAsync(ghist, 0, OS_MAXPASS * RS_BINS * sizeof(u32), st));
    const int hgrid = (int)std::min<int64_t>((count + RS_THREADS * 16 - 1) / (RS_THREADS * 16), (int64_t)ctx->num_sms * 8);
    onesweep_hist_kernel<<<hgrid, RS_THREADS, 0, st>>>(src_k, count, passes, ghist);
    KERNEL_CHECK();
    onesweep_bases_kernel<<<passes, RS_BINS, 0, st>>>(ghist);
    KERNEL_CHECK();
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)ctx->num_sms * OS_CTAS_PER_SM);
    for (int p = 0; p < passes; ++p) {
        CUDA_TRY(cudaMemsetAsync(desc, 0, desc_words * sizeof(u32), st));
        onesweep_pass_kernel<<<grid, OS_THREADS, dyn, st>>>(src_k, src_v, dst_k, dst_v, count, p * 8, tiles,
                                                           ghist + (size_t)p * RS_BINS, desc, ticket, err);
        KERNEL_CHECK();
        u64* t = src_k; src_k = dst_k; dst_k = t;
        t = src_v; src_v = dst_v; dst_v = t;
        *result_in_alt = !*result_in_alt;
    }
    return NODAL_OK;
}
